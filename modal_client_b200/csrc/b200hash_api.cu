// b200hash_api.cu -- host side of libb200hash.so: the C ABI declared in include/b200hash.h.
//
// Owns the per-device context (streams, pinned staging ring, HBM wave buffers, grow-only scratch),
// turns host batches into double-buffered waves (pack -> cudaMemcpyAsync -> trim/plan/lane_hash) and
// implements the streaming (hashlib-object shaped) interface on top of the chaining-state kernel mode.
// No CPU hashing exists in this library: without a CUDA device every entry point fails.
#include <cuda_runtime.h>
#include <stdint.h>

#include <fcntl.h>
#include <immintrin.h>
#include <pthread.h>
#include <sched.h>
#include <sys/stat.h>
#include <unistd.h>

#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cctype>
#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b200hash.h"
#include "b200hash_internal.h"
#include "b200hash_kernels.cuh"
#include "b200pack_team.h"

using namespace b200h;

static const uint32_t kShaIv[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au,
                                   0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};
static const uint32_t kMd5Iv[4] = {0x67452301u, 0xefcdab89u, 0x98badcfeu, 0x10325476u};

namespace {

thread_local std::string g_create_error;

// NVTX range around every C-ABI entry point (visible in nsys / ncu --nvtx; a no-op without an injected tool)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};
#define B200H_RANGE(name) NvtxRange nvtx_range__(name)

// One caller's small b200h_hash_batch_host request while it waits to be merged with its neighbours'.
struct CombineReq {
    const uint8_t* base;
    const uint64_t* off;
    const uint64_t* len;
    uint64_t n;
    uint32_t flags;
    uint8_t* sha;
    uint8_t* md5;
    uint64_t* trim;
    int rc = 0;
    bool done = false;
};

// Combining queue for concurrent small requests (the reference's ThreadPool / to_thread callers each hash ONE
// file, block or payload per call: py/modal/volume.py:1209-1216, blob_utils.py:622-645).  The first caller in
// becomes the leader; while it waits for the context (the GPU is busy with the previous group) the others join
// its group; the leader then issues ONE batch for all of them and hands every caller its own digests.
struct Combiner {
    std::mutex m;
    std::condition_variable cv_done, cv_more;
    std::vector<CombineReq*> pending[2];  // [B200H_TRIM_ZEROS?]: trimming changes what a message means, never mixed
    bool leader[2] = {false, false};
    bool recent_multi = false;  // the last group had company: worth waiting a moment for the next one to fill
    uint64_t groups = 0, requests = 0;
};
constexpr uint64_t kCombineMaxN = 1024;     // requests with more messages fill the GPU on their own
constexpr size_t kCombineFull = 64;          // stop waiting for company at this many callers
constexpr int kCombineWaitUs = 200;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct Wave {
    uint64_t i0, i1;    // message index range [i0, i1)
    uint64_t src_lo;    // direct mode: host offset (relative to base) of the first byte copied
    uint64_t bytes;     // bytes occupying the device wave buffer
    // A message larger than one wave slot is hashed as consecutive segments of itself (one wave each), the
    // chaining state travelling through a device-resident ChainState: seg != 0, message i0, bytes
    // [seg_start, seg_start + bytes) of it.
    int seg = 0;        // 0 = ordinary wave, 1 = first/middle segment, 2 = last segment
    bool seg_first = false;
    uint64_t seg_start = 0;
};

}  // namespace

struct b200h_ctx {
    int device = 0;
    std::mutex mu;
    std::string err;
    cudaStream_t s_copy = nullptr, s_comp = nullptr, s_chain = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // Outlier path: the warp-specialised chain kernel (TMA tile ring + mbarriers; schedule expansion, SHA-256 rounds
    // and MD5 on three warps of one CTA) runs ONE chain about twice as fast as a lane does (62 vs 30 MB/s fused),
    // at up to 4 CTAs per SM.  The planner (plan_scan_kernel) hands it only true outliers and only when all of
    // them fit in chain_cap CTAs; everything else stays on the lane kernel.  B200H_CHAIN=0 disables it, =N sets the cap.
    bool chain_enabled = true;
    // One chain CTA per SM, each hosting up to chain_groups_per_cta() messages (set from the SM count at create).
    uint32_t chain_cap = 592;
    uint32_t sm_count = 148;
    // B200H_YIELD_CHAIN_SMS=1: CTAs of a full-grid lane launch leave the SMs that host chain CTAs.  Off by default:
    // measured on one rank's share of C3 (profiles/r2_c3v2_probe.md) it moved nothing (309 vs 310 ms) -- the long pole
    // there was the lane tail, not the chains -- and it must never be applied to a small grid (see launch_lane_hash).
    bool yield_chain_sms = false;
    int* h_plan = nullptr;        // pinned: the planner's control block {avail, head, tail, outliers} of the last batch
    uint32_t last_outliers = 0;
    bool verify_plan = false;     // B200H_VERIFY_PLAN=1: cross-check the host-side outlier count against the device's
    uint64_t plan_syncs = 0;      // enqueues that had to read the outlier count back (stream synchronisation)
    Combiner combiner;
    bool combine_enabled = true;  // B200H_COMBINE=0 turns the combining queue off
    struct StreamBuf {            // resources of a b200h_stream, pooled per context (allocation costs ~1 ms)
        uint8_t* h = nullptr;     // pinned host accumulation buffer
        uint8_t* d = nullptr;     // device block: states | meta | out | plan scratch | ring | data
        cudaStream_t st = nullptr;
        cudaEvent_t ev = nullptr;
    };
    std::vector<StreamBuf> stream_pool;
    size_t stream_cap = size_t(4) << 20;  // bytes absorbed per kernel launch (B200H_STREAM_BUF)
    cudaEvent_t ev_copied[2] = {nullptr, nullptr};    // H2D of a wave slot finished
    cudaEvent_t ev_consumed[2] = {nullptr, nullptr};  // kernels reading a wave slot finished
    cudaEvent_t ev_pin[2] = {nullptr, nullptr};       // H2D out of a pinned slot finished
    cudaEvent_t ev_scratch = nullptr;                 // last use of the shared scratch buffers
    bool scratch_used = false;
    cudaEvent_t ev_dedupe = nullptr;                  // last use of the dedupe table
    bool dedupe_used = false;
    uint8_t* pin[2] = {nullptr, nullptr};
    size_t pin_cap = 0;  // per slot
    uint8_t* dwave[2] = {nullptr, nullptr};
    size_t dwave_cap = 0;  // per slot
    size_t dwave_want = 0;
    DevBuf d_off, d_len, d_order, d_order_long, d_trim, d_sha, d_md5, d_scratch, d_small, d_states, d_dedupe, d_keys, d_trimctl, d_hex;
    uint64_t* h_meta = nullptr;  // pinned: offsets then lengths
    size_t h_meta_cap = 0;       // in uint64 elements
    uint64_t launches = 0;
    std::atomic<uint64_t> staged_bytes{0};  // bytes packed / read into the pinned staging ring (the rest: DMA from source)
    bool profiling = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    double prof_ms = 0.0;
    uint64_t prof_n = 0;
    int pack_threads = 1;
    int io_threads = 1;
    PackTeam team;  // the packer / reader threads (used under `mu` only)
    // CPUs of the NUMA node the GPU hangs off (empty set: unknown / single node / B200H_NUMA=0).  The packer and
    // reader threads are pinned there: the staging ring lives in that node's memory and the DMA engine reads it from
    // there, so a packer on the other socket would push every byte across the socket interconnect twice.
    cpu_set_t node_cpus;
    bool node_cpus_valid = false;
};

struct b200h_stream {
    b200h_ctx* ctx = nullptr;
    uint32_t flags = 0;
    b200h_ctx::StreamBuf res;
    uint8_t* hbuf = nullptr;  // = res.h: pinned host accumulation buffer (cap bytes, multiple of 64)
    size_t cap = 0;
    size_t fill = 0;
    bool h2d_pending = false;      // res.ev marks the end of the last copy out of hbuf
    uint8_t* d_buf = nullptr;      // device copy of hbuf
    ChainState* d_state = nullptr; // [0] running state, [1] scratch copy for digest()
    uint64_t* d_meta = nullptr;    // off, len
    uint8_t* d_out = nullptr;      // 32 + 16
    uint32_t* d_plan = nullptr;    // this stream's own planner scratch + ring: its launches never wait for other batches
    uint32_t* d_ring = nullptr;
    uint64_t total = 0;
};

namespace {

void stream_res_destroy(b200h_ctx::StreamBuf& r);  // defined with the streaming entry points

// "0-31,64-95" -> cpu_set_t
bool parse_cpulist(const char* s, cpu_set_t* out) {
    CPU_ZERO(out);
    int n = 0;
    while (*s && *s != '\n') {
        char* end = nullptr;
        long a = strtol(s, &end, 10);
        if (end == s) return false;
        long b = a;
        if (*end == '-') {
            s = end + 1;
            b = strtol(s, &end, 10);
            if (end == s) return false;
        }
        for (long c = a; c <= b && c < CPU_SETSIZE; ++c) {
            CPU_SET((int)c, out);
            ++n;
        }
        s = *end == ',' ? end + 1 : end;
    }
    return n > 0;
}

// CPUs local to CUDA device `device` (sysfs: the PCI function's numa_node -> that node's cpulist)
bool gpu_node_cpus(int device, cpu_set_t* out) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
    char path[128], buf[4096];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return false;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    if (node < 0) return false;
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return false;
    const bool got = fgets(buf, sizeof buf, f) != nullptr;
    fclose(f);
    if (!got || !parse_cpulist(buf, out)) return false;
    // keep only CPUs this process may run on (cgroup / taskset); if none is left, give up
    cpu_set_t allowed;
    if (sched_getaffinity(0, sizeof allowed, &allowed) == 0) {
        cpu_set_t both;
        CPU_AND(&both, out, &allowed);
        if (CPU_COUNT(&both) == 0) return false;
        // a process already confined to a subset keeps its own mask
        *out = both;
    }
    return true;
}

int fail(b200h_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    else g_create_error = msg;
    return code;
}

#define CU_TRY(ctx, call)                                                                                   \
    do {                                                                                                    \
        cudaError_t e__ = (call);                                                                           \
        if (e__ != cudaSuccess) {                                                                           \
            char b__[512];                                                                                  \
            snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            cudaGetLastError();                                                                             \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? B200H_E_NOMEM : B200H_E_CUDA, b__);         \
        }                                                                                                   \
    } while (0)

int ensure_dev(b200h_ctx* ctx, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap) return 0;
    size_t want = std::max(bytes, b.cap + b.cap / 2);
    want = (want + 255) & ~size_t(255);
    if (b.p) {
        CU_TRY(ctx, cudaDeviceSynchronize());
        CU_TRY(ctx, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    CU_TRY(ctx, cudaMalloc(&b.p, want));
    b.cap = want;
    return 0;
}

int ensure_wave(b200h_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->dwave_cap) return 0;
    // grow geometrically towards the configured wave size; beyond it only as far as one message needs
    size_t want = std::max(bytes, std::min(ctx->dwave_want, std::max<size_t>(2 * ctx->dwave_cap, size_t(64) << 20)));
    want = (want + 255) & ~size_t(255);
    CU_TRY(ctx, cudaDeviceSynchronize());
    for (int s = 0; s < 2; ++s) {
        if (ctx->dwave[s]) CU_TRY(ctx, cudaFree(ctx->dwave[s]));
        ctx->dwave[s] = nullptr;
    }
    ctx->dwave_cap = 0;
    for (int s = 0; s < 2; ++s) CU_TRY(ctx, cudaMalloc(&ctx->dwave[s], want));
    ctx->dwave_cap = want;
    return 0;
}

int ensure_meta(b200h_ctx* ctx, size_t elems) {
    if (elems <= ctx->h_meta_cap) return 0;
    if (ctx->h_meta) CU_TRY(ctx, cudaFreeHost(ctx->h_meta));
    ctx->h_meta = nullptr;
    ctx->h_meta_cap = 0;
    size_t want = std::max(elems, size_t(1) << 16);
    CU_TRY(ctx, cudaHostAlloc(&ctx->h_meta, want * sizeof(uint64_t), cudaHostAllocDefault));
    ctx->h_meta_cap = want;
    return 0;
}

int prof_begin(b200h_ctx* ctx, cudaStream_t st, cudaEvent_t* a, cudaEvent_t* b) {
    *a = *b = nullptr;
    if (!ctx->profiling) return 0;
    CU_TRY(ctx, cudaEventCreate(a));
    CU_TRY(ctx, cudaEventCreate(b));
    CU_TRY(ctx, cudaEventRecord(*a, st));
    return 0;
}
int prof_end(b200h_ctx* ctx, cudaStream_t st, cudaEvent_t a, cudaEvent_t b) {
    if (!a) return 0;
    CU_TRY(ctx, cudaEventRecord(b, st));
    ctx->prof_events.emplace_back(a, b);
    return 0;
}

constexpr uint32_t kFlagNoFinal = 0x80000000u;  // internal: continuation segment (no padding, state written back)

// Enqueue trim -> plan -> lane_hash for n device-resident messages on `st`.  ctx->mu must be held.
// h_len (may be NULL) = the same lengths on the host.  With them the outlier routing is decided here without reading
// anything back, so the call only enqueues; without them (and without B200H_NO_OUTLIERS) the planner's count is
// read back after the ~12 us plan kernels, which synchronises `st` once.
int enqueue_device_batch(b200h_ctx* ctx, const uint8_t* d_base, const uint64_t* d_off, const uint64_t* d_len,
                         uint64_t n, uint32_t flags, uint8_t* d_sha, uint8_t* d_md5, uint64_t* d_trim_out,
                         ChainState* d_state, cudaStream_t st, const uint64_t* h_len = nullptr,
                         uint32_t* own_scratch = nullptr, uint32_t* own_ring = nullptr) {
    if (n == 0) return 0;
    if (n > 0xffffffffull) return fail(ctx, B200H_E_INVALID, "batch larger than 2^32-1 messages");
    uint32_t kflags = 0;
    if (flags & B200H_SHA256) kflags |= F_SHA256;
    if (flags & B200H_MD5) kflags |= F_MD5;
    if (flags & kFlagNoFinal) kflags |= F_NO_FINAL;
    if (!(kflags & (F_SHA256 | F_MD5))) return fail(ctx, B200H_E_INVALID, "flags select neither SHA256 nor MD5");

    // own_scratch / own_ring: planner scratch and queue ring private to the caller (a b200h_stream): the batch then
    // shares nothing with other batches of the context and runs concurrently with them on its own CUDA stream.
    const bool shared_scratch = own_scratch == nullptr;
    if (shared_scratch && ctx->scratch_used) CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_scratch, 0));
    const uint64_t* len_used = d_len;
    if (flags & B200H_TRIM_ZEROS) {
        uint64_t* tbuf = d_trim_out;
        if (!tbuf) {
            if (int rc = ensure_dev(ctx, ctx->d_trim, n * sizeof(uint64_t))) return rc;
            tbuf = (uint64_t*)ctx->d_trim.p;
        }
        if (int rc = ensure_dev(ctx, ctx->d_trimctl, 16 + n * sizeof(TrimWideEntry))) return rc;
        ctx->launches += launch_trim(d_base, d_off, d_len, n, tbuf, (unsigned long long*)ctx->d_trimctl.p,
                                     (TrimWideEntry*)((uint8_t*)ctx->d_trimctl.p + 16), st);
        len_used = tbuf;
        h_len = nullptr;  // the lengths that matter now exist on the device only
    } else if (d_trim_out) {
        CU_TRY(ctx, cudaMemcpyAsync(d_trim_out, d_len, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    }
    // work queue (ring + control block) and chaining-state scratch for the persistent lane kernel
    if (n >= 0x7fffffffull) return fail(ctx, B200H_E_INVALID, "batch larger than 2^31-2 messages");
    if (shared_scratch) {
        if (int rc = ensure_dev(ctx, ctx->d_order, (size_t)ring_capacity(n) * sizeof(uint32_t))) return rc;
        if (int rc = ensure_dev(ctx, ctx->d_order_long, (size_t)kLongRingCapacity * sizeof(uint32_t))) return rc;
        if (int rc = ensure_dev(ctx, ctx->d_scratch, (kPlanScratchWords + kMaxChain) * sizeof(uint32_t))) return rc;
    }
    uint32_t* ring = shared_scratch ? (uint32_t*)ctx->d_order.p : own_ring;
    // the long lane messages get a queue of their own (a private single-message batch never has any)
    // (nor does a B200H_NO_OUTLIERS batch whose lengths the host does not hold: that flag promises "only enqueues",
    // and sizing the second launch would need the planner's answer)
    uint32_t* ring_long = (shared_scratch && !((flags & B200H_NO_OUTLIERS) && !h_len)) ? (uint32_t*)ctx->d_order_long.p : nullptr;
    const uint32_t long_cap = ring_long ? plan_long_cap() : 0u;
    uint32_t* scratch = shared_scratch ? (uint32_t*)ctx->d_scratch.p : own_scratch;
    uint32_t* chain_list = scratch + kPlanScratchWords;
    int* qctl = plan_qctl(scratch);
    ChainState* states = d_state;
    if (!states) {
        if (int rc = ensure_dev(ctx, ctx->d_states, n * sizeof(ChainState))) return rc;
        states = (ChainState*)ctx->d_states.p;
    }
    const bool resume = d_state != nullptr;
    const bool chain_on = ctx->chain_enabled && !(flags & B200H_NO_OUTLIERS);
    const uint32_t max_chain = chain_on ? ctx->chain_cap : 0u;
    const uint32_t ratio8 = plan_ratio8(kflags);
    ctx->launches += launch_plan(len_used, n, ring, ring_long, chain_list, scratch, /*fresh=*/!resume, max_chain, ratio8, st);
    int* qctl_long = qctl + kLongQctlAfterQctl;
    // How many outliers did the planner pick?  The count is read back (16 bytes, one stream synchronisation after
    // the ~12 us plan kernels) because a chain kernel launched "just in case" is not free: its CTAs ask for half an
    // SM's shared memory and, idle or not, skew where the lane kernel's CTAs land (1 024 x 8 MiB: 260 -> 937 ms,
    // 2 048 x 4 MiB: 159 -> 280 ms measured with a speculative launch before / after the lane kernel).
    // So: lengths known on the host -> the same selection is computed here (plan_outliers_host); otherwise read back.
    // The same goes for the long lane queue (its launch is sized on the host as well).  A batch too small to have
    // either (nothing reaches kChainMinBlocks) needs no answer at all -- but only the host can know that.
    uint32_t n_chain = 0, n_long = 0;
    if (chain_on || long_cap) {
        const bool mirrored = h_len != nullptr;
        if (mirrored) n_chain = plan_outliers_host(h_len, n, max_chain, ctx->sm_count, long_cap, ratio8, &n_long);
        if (!mirrored || ctx->verify_plan) {
            CU_TRY(ctx, cudaMemcpyAsync(ctx->h_plan, qctl, kPlanReadbackInts * sizeof(int), cudaMemcpyDeviceToHost, st));
            CU_TRY(ctx, cudaStreamSynchronize(st));
            ctx->plan_syncs += 1;
            const uint32_t d_chain = (uint32_t)ctx->h_plan[3], d_long = (uint32_t)ctx->h_plan[kLongQctlAfterQctl + 3];
            if (mirrored && (n_chain != d_chain || n_long != d_long)) {
                char b[160];
                snprintf(b, sizeof b, "plan mismatch: host chain %u long %u, device chain %u long %u", n_chain, n_long, d_chain, d_long);
                return fail(ctx, B200H_E_STATE, b);
            }
            n_chain = d_chain;
            n_long = d_long;
        }
    }
    ctx->last_outliers = n_chain;
    if (n_chain && !shared_scratch) {
        // a private single-message batch: the chain kernel IS the batch, no side stream needed
        ctx->launches += launch_chain_hash(d_base, d_off, len_used, chain_list, qctl, kflags, d_sha, d_md5, states,
                                           resume, n_chain, st);
    } else if (n_chain) {
        // the outliers set the makespan: their CTAs go first (high-priority stream), one per SM
        CU_TRY(ctx, cudaEventRecord(ctx->ev_fork, st));
        CU_TRY(ctx, cudaStreamWaitEvent(ctx->s_chain, ctx->ev_fork, 0));
        ctx->launches += launch_chain_hash(d_base, d_off, len_used, chain_list, qctl, kflags, d_sha, d_md5, states,
                                           resume, n_chain, ctx->s_chain);
        CU_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->s_chain));
    }
    cudaEvent_t pa, pb;
    if (int rc = prof_begin(ctx, st, &pa, &pb)) return rc;
    // Lane CTAs leave the SMs that host a live chain CTA to the chains (they set the makespan) -- as long as enough SMs
    // stay chain-free for the lane work (chain CTAs sit on at most n_chain SMs, one each).
    const uint32_t lane_flags = (n_chain && n_chain <= ctx->sm_count * 3 / 4 && ctx->yield_chain_sms) ? (kflags | F_YIELD_CHAIN_SMS) : kflags;
    // the short messages (dense, time-sliced), then -- same stream -- the long ones, lane-packed at one warp per SMSP
    const uint64_t n_short = n - n_chain - n_long;
    if (n_short)
        ctx->launches += launch_lane_hash(d_base, d_off, len_used, ring, ring_capacity(n), qctl, qctl, n_short, lane_flags,
                                          d_sha, d_md5, states, st);
    if (n_long)
        ctx->launches += launch_lane_hash(d_base, d_off, len_used, ring_long, kLongRingCapacity, qctl_long, qctl, n_long,
                                          lane_flags, d_sha, d_md5, states, st);
    if (int rc = prof_end(ctx, st, pa, pb)) return rc;
    if (n_chain && shared_scratch) CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_join, 0));
    CU_TRY(ctx, cudaGetLastError());
    if (shared_scratch) {
        CU_TRY(ctx, cudaEventRecord(ctx->ev_scratch, st));
        ctx->scratch_used = true;
    }
    return 0;
}

// memcpy into the pinned staging ring with non-temporal stores (b200pack_copy.cpp: widest store the CPU has).
static inline void stream_copy(uint8_t* dst, const uint8_t* src, size_t n) { b200h_stream_copy(dst, src, n); }

// Copy the packed byte range [lo, hi) of a staged wave into dst (= pinned slot, dst[0] <-> packed byte lo).
// doff[] are the packed offsets (ascending) of messages i0..i1 inside the wave.
// Where the bytes of message i come from: host memory (base + off[i]) or a file (paths[file_of[i]] at byte
// offset off[i]).  File reads go straight into the pinned staging ring with pread -- no intermediate copy.
struct Source {
    const uint8_t* base = nullptr;
    const uint64_t* off = nullptr;
    const char* const* paths = nullptr;
    const uint64_t* file_of = nullptr;
    std::atomic<int>* io_errno = nullptr;  // first I/O failure (errno, or -1 for a short read)
    std::atomic<uint64_t>* io_file = nullptr;
};

// Copy the packed byte range [lo, hi) of a staged wave into dst (= pinned slot, dst[0] <-> packed byte lo).
// doff[] are the packed offsets (ascending) of messages i0..i1 inside the wave.
void pack_range(const Source& src, const uint64_t* len, const uint64_t* doff, uint64_t i0, uint64_t i1, uint64_t lo,
                uint64_t hi, uint8_t* dst) {
    // first message whose packed end is beyond lo
    uint64_t a = i0, b = i1;
    while (a < b) {
        const uint64_t m = (a + b) / 2;
        if (doff[m] + len[m] <= lo) a = m + 1;
        else b = m;
    }
    int fd = -1;
    uint64_t fd_file = ~0ull;
    for (uint64_t i = a; i < i1 && doff[i] < hi; ++i) {
        const uint64_t s = std::max(doff[i], lo), e = std::min(doff[i] + len[i], hi);
        if (e <= s) continue;
        if (!src.paths) {
            stream_copy(dst + (s - lo), src.base + src.off[i] + (s - doff[i]), (size_t)(e - s));
            continue;
        }
        if (src.io_errno->load(std::memory_order_relaxed)) break;
        const uint64_t f = src.file_of[i];
        if (f != fd_file) {
            if (fd >= 0) close(fd);
            fd = open(src.paths[f], O_RDONLY | O_CLOEXEC);
            fd_file = f;
        }
        int err = fd < 0 ? errno : 0;
        uint64_t got = 0;
        const uint64_t want = e - s, at = src.off[i] + (s - doff[i]);
        while (!err && got < want) {
            const ssize_t r = pread(fd, dst + (s - lo) + got, (size_t)(want - got), (off_t)(at + got));
            if (r < 0) {
                if (errno == EINTR) continue;
                err = errno;
            } else if (r == 0) {
                err = -1;  // the file is shorter than the size the caller passed
            } else {
                got += (uint64_t)r;
            }
        }
        if (err) {
            int expected = 0;
            if (src.io_errno->compare_exchange_strong(expected, err)) src.io_file->store(f);
            break;
        }
    }
    if (fd >= 0) close(fd);
}

// Fill dst with the packed byte range [lo, hi) using up to `threads` threads.  The range is cut into grains (>= 1 MiB,
// about eight per thread) that the threads take from a shared counter: with a static split the slot is only as fast as
// its slowest thread, and the packers share their cores with the DMA set-up, Python threads, a second context's team
// and, under torchrun, the other ranks' teams.  (Build machine, a shared 8-core VM, scattered 256 KiB sources into
// 256 MiB slots, best of three runs: two teams of 8 threads at once 44.6 -> 48.1 GiB/s, two teams of 16 39.6 -> 43.6,
// two teams of 4 53.0 -> 55.5; a lone team of 8 swung between 12 and 24 GiB/s with the static split and 17 and 41 with
// grains while a neighbour was busy;
// profiles/r2_stream_copy_build_machine.txt.)  The threads are the context's PackTeam; the calling thread works too.
void pack_parallel(PackTeam& team, int threads, const Source& src, const uint64_t* len, const uint64_t* doff, uint64_t i0,
                   uint64_t i1, uint64_t lo, uint64_t hi, uint8_t* dst, const cpu_set_t* cpus = nullptr) {
    const uint64_t bytes = hi - lo;
    // memory sources: one thread per >= 4 MiB; file sources: syscalls dominate small files, so also split by count
    uint64_t want = bytes / (4u << 20);
    if (src.paths) want = std::max<uint64_t>(want, (i1 - i0) / 64);
    const int t = (int)std::min<uint64_t>((uint64_t)threads, want);
    if (t <= 1) {
        pack_range(src, len, doff, i0, i1, lo, hi, dst);
        return;
    }
    const uint64_t grain = std::max<uint64_t>(uint64_t(1) << 20, (bytes / ((uint64_t)t * 8) + 4095) & ~uint64_t(4095));
    const uint64_t grains = (bytes + grain - 1) / grain;
    std::atomic<uint64_t> next{0};
    auto work = [&] {
        for (;;) {
            const uint64_t g = next.fetch_add(1, std::memory_order_relaxed);
            if (g >= grains) return;
            const uint64_t a = lo + g * grain, b = std::min(hi, a + grain);
            pack_range(src, len, doff, i0, i1, a, b, dst + (a - lo));
        }
    };
    team.run(t, cpus, work);
}

// A sparse selection of page-locked memory whose messages average at least this many bytes is DMAed one message at a
// time (gather_pinned): one cudaMemcpyAsync costs a few microseconds, a 1 MiB message ~20 us of PCIe.
constexpr uint64_t kGatherMinAvg = uint64_t(1) << 20;

int hash_batch_host_impl(b200h_ctx* ctx, const uint8_t* base, const uint64_t* off, const uint64_t* len, uint64_t n,
                         uint32_t flags, uint8_t* sha_out, uint8_t* md5_out, uint64_t* trim_out, uint8_t* etag_out,
                         const char* const* paths = nullptr, const uint64_t* file_of = nullptr,
                         bool gather_pinned = false) {
    if (n == 0) return 0;
    std::atomic<int> io_errno{0};
    std::atomic<uint64_t> io_file{0};
    Source src;
    src.base = base;
    src.off = off;
    src.paths = paths;
    src.file_of = file_of;
    src.io_errno = &io_errno;
    src.io_file = &io_file;
    if (!off || !len) return fail(ctx, B200H_E_INVALID, "offsets/lengths must not be NULL");
    if (!(flags & (B200H_SHA256 | B200H_MD5))) return fail(ctx, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    if (etag_out && !(flags & B200H_MD5)) return fail(ctx, B200H_E_INVALID, "etag requires B200H_MD5");
    CU_TRY(ctx, cudaSetDevice(ctx->device));

    // Page-locked source?  Then DMA straight from the caller's memory, no staging copy.
    // (Only when the messages cover most of the span they sit in: a wave DMAs its whole [min offset, max end) span,
    // so a sparse selection -- one rank's interleaved shard of a shared buffer -- would copy the gaps too; those
    // are gathered through the staging ring like pageable memory.)
    // (gather_pinned: a device group member's share, dealt from the whole batch, is sparse by construction; large
    // messages are then DMAed one by one into the packed wave layout instead.)
    bool direct = false, gather = false;
    if (base && !paths) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, base) == cudaSuccess) direct = (at.type == cudaMemoryTypeHost);
        else cudaGetLastError();
        if (direct) {
            uint64_t lo = ~0ull, hi = 0, payload = 0;
            for (uint64_t i = 0; i < n; ++i) {
                lo = std::min(lo, off[i]);
                hi = std::max(hi, off[i] + len[i]);
                payload += len[i];
            }
            if (hi - lo > payload + payload / 4 + (uint64_t(16) << 20))
                direct = gather = gather_pinned && payload >= n * kGatherMinAvg;
        }
    }

    if (int rc = ensure_meta(ctx, 2 * n)) return rc;
    uint64_t* doff = ctx->h_meta;      // device-relative offsets
    uint64_t* hlen = ctx->h_meta + n;  // lengths (pinned copy)
    memcpy(hlen, len, n * sizeof(uint64_t));

    // ---- carve the batch into waves that fit one HBM wave slot
    size_t cap = std::max(ctx->dwave_cap, ctx->dwave_want);
    const uint64_t seg_cap = cap & ~uint64_t(63);
    std::vector<Wave> waves;
    {
        uint64_t i = 0;
        while (i < n) {
            Wave w{i, i, 0, 0};
            if (len[i] + 16 > cap) {
                // oversized message: consecutive 64-byte-aligned segments, one wave each
                if (flags & B200H_TRIM_ZEROS)
                    return fail(ctx, B200H_E_INVALID, "B200H_TRIM_ZEROS is not supported for a message larger than one staging wave");
                for (uint64_t s0 = 0; s0 < len[i]; s0 += seg_cap) {
                    Wave sw{i, i + 1, 0, std::min<uint64_t>(seg_cap, len[i] - s0)};
                    sw.seg = (s0 + seg_cap >= len[i]) ? 2 : 1;
                    sw.seg_first = s0 == 0;
                    sw.seg_start = s0;
                    waves.push_back(sw);
                }
                doff[i] = 0;
                i += 1;
                continue;
            }
            if (direct && !gather) {
                uint64_t lo = off[i], hi = off[i] + len[i];
                uint64_t j = i + 1;
                for (; j < n; ++j) {
                    if (len[j] + 16 > cap) break;  // oversized: gets its own segment waves
                    const uint64_t nlo = std::min(lo, off[j]), nhi = std::max(hi, off[j] + len[j]);
                    if (nhi - (nlo & ~15ull) > cap) break;
                    lo = nlo;
                    hi = nhi;
                }
                w.i1 = j;
                w.src_lo = lo & ~15ull;  // keep the 16-byte phase of every message
                w.bytes = hi - w.src_lo;
                for (uint64_t k = i; k < j; ++k) doff[k] = off[k] - w.src_lo;
            } else {
                uint64_t used = 0;
                uint64_t j = i;
                for (; j < n; ++j) {
                    const uint64_t need = (len[j] + 15) & ~15ull;
                    if (len[j] + 16 > cap) break;  // oversized: gets its own segment waves
                    if (j > i && used + need > cap) break;
                    doff[j] = used;
                    used += need;
                }
                w.i1 = j;
                w.bytes = used;
            }
            waves.push_back(w);
            i = w.i1;
        }
    }
    size_t need_wave = 16;
    for (auto& w : waves) need_wave = std::max<size_t>(need_wave, w.bytes);
    if (int rc = ensure_wave(ctx, need_wave)) return rc;

    if (int rc = ensure_dev(ctx, ctx->d_off, n * sizeof(uint64_t))) return rc;
    if (int rc = ensure_dev(ctx, ctx->d_len, n * sizeof(uint64_t))) return rc;
    if (int rc = ensure_dev(ctx, ctx->d_trim, n * sizeof(uint64_t))) return rc;
    if (flags & B200H_SHA256)
        if (int rc = ensure_dev(ctx, ctx->d_sha, n * 32)) return rc;
    if (flags & B200H_MD5)
        if (int rc = ensure_dev(ctx, ctx->d_md5, n * 16 + 16)) return rc;
    uint64_t* d_off = (uint64_t*)ctx->d_off.p;
    uint64_t* d_len = (uint64_t*)ctx->d_len.p;
    uint64_t* d_trim = (uint64_t*)ctx->d_trim.p;
    uint8_t* d_sha = (flags & B200H_SHA256) ? (uint8_t*)ctx->d_sha.p : nullptr;
    uint8_t* d_md5 = (flags & B200H_MD5) ? (uint8_t*)ctx->d_md5.p : nullptr;

    CU_TRY(ctx, cudaMemcpyAsync(d_off, doff, n * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->s_comp));
    CU_TRY(ctx, cudaMemcpyAsync(d_len, hlen, n * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->s_comp));

    if (int rc = ensure_dev(ctx, ctx->d_small, 256)) return rc;
    uint64_t* d_segmeta = (uint64_t*)((uint8_t*)ctx->d_small.p + 64);
    ChainState* d_segstate = (ChainState*)((uint8_t*)ctx->d_small.p + 128);

    bool pin_used[2] = {false, false};
    int pin_slot = 0;
    for (size_t wi = 0; wi < waves.size(); ++wi) {
        const Wave& w = waves[wi];
        const int slot = (int)(wi & 1);
        if (wi >= 2) CU_TRY(ctx, cudaStreamWaitEvent(ctx->s_copy, ctx->ev_consumed[slot], 0));
        // a segment wave is message w.i0 restricted to [seg_start, seg_start + bytes), placed at device offset 0
        const uint64_t seg_off1 = w.seg ? off[w.i0] + w.seg_start : 0, seg_len1 = w.bytes, seg_doff1 = 0;
        const uint64_t seg_file1 = (w.seg && file_of) ? file_of[w.i0] : 0;
        Source seg_src = src;
        seg_src.off = &seg_off1;
        seg_src.file_of = file_of ? &seg_file1 : nullptr;
        if (gather && !w.seg) {
            for (uint64_t k = w.i0; k < w.i1; ++k)
                if (len[k])
                    CU_TRY(ctx, cudaMemcpyAsync(ctx->dwave[slot] + doff[k], base + off[k], len[k], cudaMemcpyHostToDevice,
                                                ctx->s_copy));
        } else if (direct) {
            const uint8_t* from = w.seg ? base + off[w.i0] + w.seg_start : base + w.src_lo;
            if (w.bytes) CU_TRY(ctx, cudaMemcpyAsync(ctx->dwave[slot], from, w.bytes, cudaMemcpyHostToDevice, ctx->s_copy));
        } else {
            for (uint64_t lo = 0; lo < w.bytes; lo += ctx->pin_cap) {
                const uint64_t hi = std::min<uint64_t>(w.bytes, lo + ctx->pin_cap);
                if (pin_used[pin_slot]) CU_TRY(ctx, cudaEventSynchronize(ctx->ev_pin[pin_slot]));
                const cpu_set_t* cpus = ctx->node_cpus_valid ? &ctx->node_cpus : nullptr;
                if (w.seg)
                    pack_parallel(ctx->team, paths ? ctx->io_threads : ctx->pack_threads, seg_src, &seg_len1, &seg_doff1, 0, 1, lo, hi,
                                  ctx->pin[pin_slot], cpus);
                else
                    pack_parallel(ctx->team, paths ? ctx->io_threads : ctx->pack_threads, src, len, doff, w.i0, w.i1, lo, hi,
                                  ctx->pin[pin_slot], cpus);
                if (io_errno.load()) {
                    const int e = io_errno.load();
                    CU_TRY(ctx, cudaDeviceSynchronize());
                    return fail(ctx, B200H_E_IO,
                                std::string("reading ") + paths[io_file.load()] + ": " +
                                    (e == -1 ? "file is shorter than the size passed in" : strerror(e)));
                }
                CU_TRY(ctx, cudaMemcpyAsync(ctx->dwave[slot] + lo, ctx->pin[pin_slot], hi - lo, cudaMemcpyHostToDevice,
                                            ctx->s_copy));
                ctx->staged_bytes += hi - lo;
                CU_TRY(ctx, cudaEventRecord(ctx->ev_pin[pin_slot], ctx->s_copy));
                pin_used[pin_slot] = true;
                pin_slot ^= 1;
            }
        }
        CU_TRY(ctx, cudaEventRecord(ctx->ev_copied[slot], ctx->s_copy));
        CU_TRY(ctx, cudaStreamWaitEvent(ctx->s_comp, ctx->ev_copied[slot], 0));
        const uint64_t cnt = w.i1 - w.i0;
        if (w.seg) {
            if (w.seg_first) {
                ChainState iv;
                memcpy(iv.sha, kShaIv, sizeof kShaIv);
                memcpy(iv.md5, kMd5Iv, sizeof kMd5Iv);
                iv.prior_bytes = 0;
                iv.reserved = 0;
                CU_TRY(ctx, cudaMemcpyAsync(d_segstate, &iv, sizeof iv, cudaMemcpyHostToDevice, ctx->s_comp));
            }
            const uint64_t meta[2] = {0, w.bytes};
            CU_TRY(ctx, cudaMemcpyAsync(d_segmeta, meta, sizeof meta, cudaMemcpyHostToDevice, ctx->s_comp));
            const uint32_t f = (flags & (3u | B200H_NO_OUTLIERS)) | (w.seg == 2 ? 0u : kFlagNoFinal);
            const uint64_t seg_bytes = w.bytes;
            if (int rc = enqueue_device_batch(ctx, ctx->dwave[slot], d_segmeta, d_segmeta + 1, 1, f,
                                              d_sha ? d_sha + 32 * w.i0 : nullptr, d_md5 ? d_md5 + 16 * w.i0 : nullptr,
                                              nullptr, d_segstate, ctx->s_comp, &seg_bytes))
                return rc;
            if (w.seg == 2)
                CU_TRY(ctx, cudaMemcpyAsync(d_trim + w.i0, d_len + w.i0, sizeof(uint64_t), cudaMemcpyDeviceToDevice, ctx->s_comp));
            CU_TRY(ctx, cudaEventRecord(ctx->ev_consumed[slot], ctx->s_comp));
            continue;
        }
        if (int rc = enqueue_device_batch(ctx, ctx->dwave[slot], d_off + w.i0, d_len + w.i0, cnt, flags,
                                          d_sha ? d_sha + 32 * w.i0 : nullptr, d_md5 ? d_md5 + 16 * w.i0 : nullptr,
                                          d_trim + w.i0, nullptr, ctx->s_comp, len + w.i0))
            return rc;
        CU_TRY(ctx, cudaEventRecord(ctx->ev_consumed[slot], ctx->s_comp));
    }

    uint8_t* d_etag = nullptr;
    if (etag_out) {
        // MD5 over the concatenated raw part digests, still on the device (blob_utils.py:216-219)
        if (int rc = ensure_dev(ctx, ctx->d_small, 64)) return rc;
        uint64_t meta[2] = {0, n * 16};
        uint64_t* d_meta = (uint64_t*)ctx->d_small.p;
        d_etag = (uint8_t*)ctx->d_small.p + 32;
        CU_TRY(ctx, cudaMemcpyAsync(d_meta, meta, sizeof meta, cudaMemcpyHostToDevice, ctx->s_comp));
        if (int rc = enqueue_device_batch(ctx, d_md5, d_meta, d_meta + 1, 1, B200H_MD5, nullptr, d_etag, nullptr,
                                          nullptr, ctx->s_comp, &meta[1]))
            return rc;
    }
    // The output arrays may live in host OR device memory (cudaMemcpyDefault): a caller that goes on to all-gather
    // the table over NCCL passes device buffers and the digests never visit the host.
    if (flags & B200H_HEX_OUT) {
        // the digest columns leave the device as lowercase ASCII hex (64 / 32 characters per row)
        const bool want_sha = sha_out && d_sha, want_md5 = md5_out && d_md5;
        if (int rc = ensure_dev(ctx, ctx->d_hex, n * 96 + 64)) return rc;
        uint8_t* hex_sha = (uint8_t*)ctx->d_hex.p;
        uint8_t* hex_md5 = hex_sha + n * 64;
        if (want_sha) {
            ctx->launches += launch_hex_rows(d_sha, n * 32, hex_sha, ctx->s_comp);
            CU_TRY(ctx, cudaMemcpyAsync(sha_out, hex_sha, n * 64, cudaMemcpyDefault, ctx->s_comp));
        }
        if (want_md5) {
            ctx->launches += launch_hex_rows(d_md5, n * 16, hex_md5, ctx->s_comp);
            CU_TRY(ctx, cudaMemcpyAsync(md5_out, hex_md5, n * 32, cudaMemcpyDefault, ctx->s_comp));
        }
        CU_TRY(ctx, cudaGetLastError());
    } else {
        if (sha_out && d_sha) CU_TRY(ctx, cudaMemcpyAsync(sha_out, d_sha, n * 32, cudaMemcpyDefault, ctx->s_comp));
        if (md5_out && d_md5) CU_TRY(ctx, cudaMemcpyAsync(md5_out, d_md5, n * 16, cudaMemcpyDefault, ctx->s_comp));
    }
    if (trim_out) CU_TRY(ctx, cudaMemcpyAsync(trim_out, d_trim, n * sizeof(uint64_t), cudaMemcpyDefault, ctx->s_comp));
    if (etag_out) CU_TRY(ctx, cudaMemcpyAsync(etag_out, d_etag, 16, cudaMemcpyDefault, ctx->s_comp));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->s_comp));
    return 0;
}

constexpr uint32_t kPublicFlags = 7u | B200H_NO_OUTLIERS | B200H_HEX_OUT;

// A small request from one of possibly many concurrent callers: merge it with whatever else arrives while the context
// is busy, run ONE batch, hand every caller its rows.  (See Combiner.)
int combined_hash_batch_host(b200h_ctx* ctx, const uint8_t* base, const uint64_t* off, const uint64_t* len, uint64_t n,
                             uint32_t flags, uint8_t* sha_out, uint8_t* md5_out, uint64_t* trim_out) {
    Combiner& cb = ctx->combiner;
    CombineReq r{base, off, len, n, flags, sha_out, md5_out, trim_out};
    const int k = (flags & B200H_TRIM_ZEROS) ? 1 : 0;
    std::unique_lock<std::mutex> cl(cb.m);
    cb.pending[k].push_back(&r);
    if (cb.leader[k]) {  // somebody is already collecting this group: ride along
        cb.cv_more.notify_one();
        cb.cv_done.wait(cl, [&] { return r.done; });
        return r.rc;
    }
    cb.leader[k] = true;
    if (cb.recent_multi && cb.pending[k].size() < kCombineFull)  // concurrent callers were seen a moment ago
        cb.cv_more.wait_for(cl, std::chrono::microseconds(kCombineWaitUs), [&] { return cb.pending[k].size() >= kCombineFull; });
    cl.unlock();
    std::unique_lock<std::mutex> gl(ctx->mu);  // while the previous group occupies the GPU, callers keep joining this one
    cl.lock();
    std::vector<CombineReq*> grp;
    grp.swap(cb.pending[k]);
    cb.leader[k] = false;
    cb.recent_multi = grp.size() > 1;
    cb.groups += 1;
    cb.requests += grp.size();
    cl.unlock();

    int rc = 0;
    if (grp.size() == 1) {
        rc = hash_batch_host_impl(ctx, base, off, len, n, flags, sha_out, md5_out, trim_out, nullptr);
        gl.unlock();
    } else {
        uint64_t total = 0;
        uint32_t uflags = 0;
        for (CombineReq* q : grp) {
            total += q->n;
            uflags |= q->flags;
        }
        std::vector<uint64_t> aoff(total), alen(total), ttrim(total);
        std::vector<uint8_t> tsha((uflags & B200H_SHA256) ? total * 32 : 0), tmd5((uflags & B200H_MD5) ? total * 16 : 0);
        uint64_t at = 0;
        for (CombineReq* q : grp)
            for (uint64_t i = 0; i < q->n; ++i, ++at) {
                aoff[at] = (uint64_t)(uintptr_t)q->base + q->off[i];  // absolute addresses, base = NULL
                alen[at] = q->len[i];
            }
        rc = total ? hash_batch_host_impl(ctx, nullptr, aoff.data(), alen.data(), total, uflags,
                                          tsha.empty() ? nullptr : tsha.data(), tmd5.empty() ? nullptr : tmd5.data(),
                                          ttrim.data(), nullptr)
                   : 0;
        gl.unlock();
        at = 0;
        for (CombineReq* q : grp) {
            if (!rc) {
                if (q->sha && (q->flags & B200H_SHA256)) memcpy(q->sha, tsha.data() + at * 32, q->n * 32);
                if (q->md5 && (q->flags & B200H_MD5)) memcpy(q->md5, tmd5.data() + at * 16, q->n * 16);
                if (q->trim) memcpy(q->trim, ttrim.data() + at, q->n * sizeof(uint64_t));
            }
            at += q->n;
        }
    }
    cl.lock();
    for (CombineReq* q : grp) {
        q->rc = rc;
        q->done = true;
    }
    cb.cv_done.notify_all();
    return rc;
}

}  // namespace

// =============================================================================================== C ABI

extern "C" {

const char* b200h_version(void) { return kernel_build_info(); }

int b200h_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char* b200h_last_error(b200h_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int b200h_create(int device, size_t pinned_bytes, size_t device_bytes, b200h_ctx** out) {
    return b200h::create_member(device, pinned_bytes, device_bytes, nullptr, 0, out);
}

}  // extern "C"

int b200h::create_member(int device, size_t pinned_bytes, size_t device_bytes, const int* group_devices, int ngroup,
                         b200h_ctx** out) {
    if (!out) return fail(nullptr, B200H_E_INVALID, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, B200H_E_CUDA,
                    std::string("no usable CUDA device (libb200hash has no CPU fallback): ") + cudaGetErrorString(e));
    }
    if (device < 0 || device >= ndev) return fail(nullptr, B200H_E_INVALID, "device index out of range");
    b200h_ctx* ctx = new (std::nothrow) b200h_ctx();
    if (!ctx) return fail(nullptr, B200H_E_NOMEM, "out of host memory");
    ctx->device = device;
    auto bail = [&](int rc) {
        g_create_error = ctx->err;
        b200h_destroy(ctx);
        return rc;
    };
#define CU_INIT(call)                                                                              \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            ctx->err = std::string(#call " failed: ") + cudaGetErrorString(e__);                   \
            cudaGetLastError();                                                                    \
            return bail(e__ == cudaErrorMemoryAllocation ? B200H_E_NOMEM : B200H_E_CUDA);          \
        }                                                                                          \
    } while (0)
    CU_INIT(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_INIT(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        ctx->err = "device is not Blackwell-class (kernels are built for sm_100a only)";
        return bail(B200H_E_CUDA);
    }
    CU_INIT(configure_kernels());
    ctx->chain_cap = (uint32_t)std::min<long>((long)prop.multiProcessorCount * chain_groups_per_cta(), (long)kMaxChain);
    ctx->sm_count = (uint32_t)prop.multiProcessorCount;
    if (const char* e = getenv("B200H_YIELD_CHAIN_SMS")) ctx->yield_chain_sms = atoi(e) != 0;
    CU_INIT(cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking));
    CU_INIT(cudaStreamCreateWithFlags(&ctx->s_comp, cudaStreamNonBlocking));
    {
        int lo = 0, hi = 0;
        CU_INIT(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CU_INIT(cudaStreamCreateWithPriority(&ctx->s_chain, cudaStreamNonBlocking, hi));
    }
    CU_INIT(cudaHostAlloc(&ctx->h_plan, 64, cudaHostAllocDefault));
    CU_INIT(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CU_INIT(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    if (const char* e = getenv("B200H_CHAIN")) {  // tuning knob: 0 disables the outlier path, N >= 2 sets the CTA cap
        const long v = atol(e);
        ctx->chain_enabled = v > 0;
        if (v > 1) ctx->chain_cap = (uint32_t)std::min<long>(v, (long)ctx->chain_cap);  // never above groups x SMs
    }
    for (int s = 0; s < 2; ++s) {
        CU_INIT(cudaEventCreateWithFlags(&ctx->ev_copied[s], cudaEventDisableTiming));
        CU_INIT(cudaEventCreateWithFlags(&ctx->ev_consumed[s], cudaEventDisableTiming));
        CU_INIT(cudaEventCreateWithFlags(&ctx->ev_pin[s], cudaEventDisableTiming));
    }
    CU_INIT(cudaEventCreateWithFlags(&ctx->ev_scratch, cudaEventDisableTiming));
    CU_INIT(cudaEventCreateWithFlags(&ctx->ev_dedupe, cudaEventDisableTiming));
    if (pinned_bytes == 0) pinned_bytes = size_t(512) << 20;
    if (device_bytes == 0) device_bytes = size_t(8) << 30;
    ctx->pin_cap = std::max<size_t>((pinned_bytes / 2) & ~size_t(4095), 1 << 20);
    ctx->dwave_want = std::max<size_t>((device_bytes / 2) & ~size_t(255), 1 << 20);
    for (int s = 0; s < 2; ++s) CU_INIT(cudaHostAlloc(&ctx->pin[s], ctx->pin_cap, cudaHostAllocDefault));
    unsigned hc = std::thread::hardware_concurrency();
    {
        const char* e = getenv("B200H_NUMA");
        if (!(e && atoi(e) == 0)) ctx->node_cpus_valid = gpu_node_cpus(device, &ctx->node_cpus);
    }
    // One process per GPU shares the host with its siblings.  The packers run on the GPU's NUMA node, so what a rank
    // may use is that node's CPUs divided by the ranks whose GPUs hang off the same node (LOCAL_WORLD_SIZE ranks spread
    // over the nodes), and a caller that keeps two batches in flight (the map pump) runs two packer teams at once:
    // 8 ranks x 2 x 16 packers were 256 threads on 128 CPUs in the first 8-GPU run of the pump (profiles/r2_scaling.md).
    unsigned share = ctx->node_cpus_valid ? (unsigned)CPU_COUNT(&ctx->node_cpus) : hc;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) {
        const int lw = atoi(e);
        if (lw > 1) {
            unsigned nodes = 0;
            if (ctx->node_cpus_valid) {
                for (int k = 0; k < 64; ++k) {
                    char path[64];
                    snprintf(path, sizeof path, "/sys/devices/system/node/node%d", k);
                    if (access(path, F_OK) == 0) ++nodes;
                }
            }
            const unsigned per_node = nodes ? ((unsigned)lw + nodes - 1) / nodes : (unsigned)lw;
            share = std::max(4u, share / std::max(1u, per_node));
        }
    }
    // The members of a device group that sit on this device's NUMA node (this one included) divide its CPUs the same
    // way; without a known node every member shares the whole host.
    if (ngroup > 1) {
        unsigned sharers = 0;
        for (int g = 0; g < ngroup; ++g) {
            cpu_set_t other;
            if (!ctx->node_cpus_valid || group_devices[g] == device ||
                (gpu_node_cpus(group_devices[g], &other) && CPU_EQUAL(&other, &ctx->node_cpus)))
                ++sharers;
        }
        share = std::max(4u, share / std::max(1u, sharers));
    }
    ctx->pack_threads = (int)std::min(16u, std::max(2u, share / 2));  // 16: measured best on 2x Xeon 8562Y+ (8..64 tried)
    if (const char* e = getenv("B200H_PACK_THREADS")) ctx->pack_threads = std::max(1, atoi(e));
    ctx->io_threads = (int)std::min(16u, std::max(1u, share));  // measured: 16 > 32 > 64 > 128 (kernel-side contention)
    if (const char* e = getenv("B200H_IO_THREADS")) ctx->io_threads = std::max(1, atoi(e));
    if (const char* e = getenv("B200H_VERIFY_PLAN")) ctx->verify_plan = atoi(e) != 0;
    if (const char* e = getenv("B200H_COMBINE")) ctx->combine_enabled = atoi(e) != 0;
    if (const char* e = getenv("B200H_STREAM_BUF")) {
        const long long v = atoll(e);
        if (v >= 65536) ctx->stream_cap = (size_t)v & ~size_t(63);
    }
#undef CU_INIT
    *out = ctx;
    return 0;
}

void b200h::file_messages(const uint64_t* sizes, uint64_t n, uint64_t part_len, std::vector<uint64_t>& off,
                          std::vector<uint64_t>& len, std::vector<uint64_t>& file_of) {
    for (uint64_t f = 0; f < n; ++f) {
        if (part_len == 0) {
            off.push_back(0);
            len.push_back(sizes[f]);
            file_of.push_back(f);
        } else {
            for (uint64_t o = 0; o < sizes[f]; o += part_len) {
                off.push_back(o);
                len.push_back(std::min(part_len, sizes[f] - o));
                file_of.push_back(f);
            }
        }
    }
}

uint64_t b200h::staged_bytes(b200h_ctx* ctx) { return ctx->staged_bytes.load(); }

int b200h::hash_share(b200h_ctx* ctx, const uint8_t* base, const uint64_t* off, const uint64_t* len, uint64_t n,
                      uint32_t flags, uint8_t* sha_out, uint8_t* md5_out, uint64_t* trim_out, const char* const* paths,
                      const uint64_t* file_of, uint64_t* staged_out) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    const uint64_t staged0 = ctx->staged_bytes;
    const int rc = hash_batch_host_impl(ctx, base, off, len, n, flags & kPublicFlags, sha_out, md5_out, trim_out, nullptr,
                                        paths, file_of, /*gather_pinned=*/true);
    *staged_out = ctx->staged_bytes - staged0;
    return rc;
}

int b200h::ctx_device(b200h_ctx* ctx) { return ctx->device; }

int b200h::ctx_fail(b200h_ctx* ctx, int code, const std::string& msg) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    return fail(ctx, code, msg);
}

int b200h::hash_device_rows(b200h_ctx* ctx, const uint64_t* addr, const uint64_t* len, uint64_t rows, uint32_t flags,
                            uint8_t* sha_out, uint8_t* md5_out, uint64_t* trim_out, const uint64_t* row_of, uint64_t n,
                            uint8_t* etag_out, const GatherRows* gather) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    flags &= kPublicFlags;
    if (!(flags & (B200H_SHA256 | B200H_MD5))) return fail(ctx, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    if (etag_out && !(flags & B200H_MD5)) return fail(ctx, B200H_E_INVALID, "etag requires B200H_MD5");
    const uint64_t ne = etag_out ? n : 0;
    if (rows == 0 && ne == 0) return 0;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    // Gathered rows: windows of rows (one, unless the gathered bytes pass the cap), a scratch buffer as large as the
    // largest window, and the work items of gather_pieces_kernel (pieces split at gather_item_bytes), window-major.
    std::vector<uint64_t> win{0, rows}, dst, win_bytes{0}, win_items{0, 0};
    uint64_t items = 0, scratch_bytes = 0;
    if (gather) {
        gather_windows(len, gather->piece_of, rows, gather->window_bytes, win, dst, win_bytes);
        win_items.assign(1, 0);
        const uint64_t step = gather_item_bytes();
        for (size_t w = 0; w + 1 < win.size(); ++w) {
            for (uint64_t r = win[w]; r < win[w + 1]; ++r)
                for (uint64_t p = gather->piece_of[r]; p < gather->piece_of[r + 1]; ++p) items += (gather->plen[p] + step - 1) / step;
            win_items.push_back(items);
            scratch_bytes = std::max(scratch_bytes, win_bytes[w]);
        }
    }
    struct Scratch {
        void* p = nullptr;
        ~Scratch() {
            if (p) cudaFree(p);
        }
    } scratch;
    if (scratch_bytes) {
        const cudaError_t e = cudaMalloc(&scratch.p, scratch_bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            scratch.p = nullptr;
            return fail(ctx, e == cudaErrorMemoryAllocation ? B200H_E_NOMEM : B200H_E_CUDA,
                        "cannot allocate " + std::to_string(scratch_bytes) + " bytes of gather scratch on cuda:" +
                            std::to_string(ctx->device) + " (" + cudaGetErrorString(e) + ")");
        }
    }
    // One pinned table -- addresses | lengths | ETag segment offsets | ETag segment lengths | gather sources |
    // gather destinations | gather lengths -- and one copy of it.
    // A zero-length row reads nothing; it is pointed at library scratch so that no kernel ever sees a stray address.
    if (int rc = ensure_meta(ctx, 2 * rows + 2 * ne + 3 * items)) return rc;
    if (int rc = ensure_dev(ctx, ctx->d_small, 256)) return rc;
    uint64_t* h = ctx->h_meta;
    for (uint64_t i = 0; i < rows; ++i) {
        const bool gathered = gather && gather->piece_of[i + 1] > gather->piece_of[i];
        h[i] = !len[i] ? (uint64_t)(uintptr_t)ctx->d_small.p : gathered ? (uint64_t)(uintptr_t)scratch.p + dst[i] : addr[i];
        h[rows + i] = len[i];
    }
    for (uint64_t b = 0; b < ne; ++b) {
        h[2 * rows + b] = 16 * row_of[b];
        h[2 * rows + ne + b] = 16 * (row_of[b + 1] - row_of[b]);
    }
    uint64_t* h_items = h + 2 * rows + 2 * ne;
    if (items) {
        const uint64_t step = gather_item_bytes();
        uint64_t t = 0;
        for (uint64_t r = 0; r < rows; ++r) {
            uint64_t at = h[r];  // the row's place in scratch; its pieces follow one another there
            for (uint64_t p = gather->piece_of[r]; p < gather->piece_of[r + 1]; at += gather->plen[p++])
                for (uint64_t o = 0; o < gather->plen[p]; o += step, ++t) {
                    h_items[t] = gather->psrc[p] + o;
                    h_items[items + t] = at + o;
                    h_items[2 * items + t] = std::min(step, gather->plen[p] - o);
                }
        }
    }
    const size_t table_bytes = (2 * rows + 2 * ne + 3 * items) * sizeof(uint64_t);
    if (int rc = ensure_dev(ctx, ctx->d_off, table_bytes)) return rc;
    if (int rc = ensure_dev(ctx, ctx->d_trim, rows * sizeof(uint64_t) + 8)) return rc;
    if (flags & B200H_SHA256)
        if (int rc = ensure_dev(ctx, ctx->d_sha, rows * 32 + 32)) return rc;
    if (flags & B200H_MD5)
        if (int rc = ensure_dev(ctx, ctx->d_md5, rows * 16 + 16)) return rc;
    // d_hex: hex SHA-256 rows | hex MD5 rows | ETags (16-byte aligned: rows * 96)
    if (int rc = ensure_dev(ctx, ctx->d_hex, rows * 96 + ne * 16 + 64)) return rc;
    uint64_t* d_tab = (uint64_t*)ctx->d_off.p;
    uint64_t* d_trim = (uint64_t*)ctx->d_trim.p;
    uint8_t* d_sha = (flags & B200H_SHA256) ? (uint8_t*)ctx->d_sha.p : nullptr;
    uint8_t* d_md5 = (flags & B200H_MD5) ? (uint8_t*)ctx->d_md5.p : nullptr;
    uint8_t* hex_sha = (uint8_t*)ctx->d_hex.p;
    uint8_t* hex_md5 = hex_sha + rows * 64;
    uint8_t* d_etag = hex_sha + rows * 96;
    CU_TRY(ctx, cudaMemcpyAsync(d_tab, h, table_bytes, cudaMemcpyHostToDevice, ctx->s_comp));
    // the lengths are known here: outliers are routed without a read-back (B200H_TRIM_ZEROS still needs its one)
    const uint64_t* d_items = d_tab + 2 * rows + 2 * ne;
    for (size_t w = 0; w + 1 < win.size(); ++w) {
        const uint64_t r0 = win[w], nr = win[w + 1] - win[w], i0 = win_items[w], ni = win_items[w + 1] - win_items[w];
        if (ni) {
            ctx->launches += launch_gather(d_items + i0, d_items + items + i0, d_items + 2 * items + i0, ni, ctx->s_comp);
            CU_TRY(ctx, cudaGetLastError());
        }
        if (nr)
            if (int rc = enqueue_device_batch(ctx, nullptr, d_tab + r0, d_tab + rows + r0, nr, flags,
                                              d_sha ? d_sha + 32 * r0 : nullptr, d_md5 ? d_md5 + 16 * r0 : nullptr,
                                              d_trim + r0, nullptr, ctx->s_comp, len + r0))
                return rc;
    }
    if (ne)
        // every buffer's ETag in one batch: message b = its segment of the raw MD5 table (blob_utils.py:216-219)
        if (int rc = enqueue_device_batch(ctx, d_md5, d_tab + 2 * rows, d_tab + 2 * rows + ne, ne, B200H_MD5, nullptr,
                                          d_etag, nullptr, nullptr, ctx->s_comp, h + 2 * rows + ne))
            return rc;
    if (flags & B200H_HEX_OUT) {
        if (sha_out && d_sha && rows) {
            ctx->launches += launch_hex_rows(d_sha, rows * 32, hex_sha, ctx->s_comp);
            CU_TRY(ctx, cudaMemcpyAsync(sha_out, hex_sha, rows * 64, cudaMemcpyDefault, ctx->s_comp));
        }
        if (md5_out && d_md5 && rows) {
            ctx->launches += launch_hex_rows(d_md5, rows * 16, hex_md5, ctx->s_comp);
            CU_TRY(ctx, cudaMemcpyAsync(md5_out, hex_md5, rows * 32, cudaMemcpyDefault, ctx->s_comp));
        }
        CU_TRY(ctx, cudaGetLastError());
    } else if (rows) {
        if (sha_out && d_sha) CU_TRY(ctx, cudaMemcpyAsync(sha_out, d_sha, rows * 32, cudaMemcpyDefault, ctx->s_comp));
        if (md5_out && d_md5) CU_TRY(ctx, cudaMemcpyAsync(md5_out, d_md5, rows * 16, cudaMemcpyDefault, ctx->s_comp));
    }
    if (trim_out && rows) CU_TRY(ctx, cudaMemcpyAsync(trim_out, d_trim, rows * sizeof(uint64_t), cudaMemcpyDefault, ctx->s_comp));
    if (ne) CU_TRY(ctx, cudaMemcpyAsync(etag_out, d_etag, ne * 16, cudaMemcpyDefault, ctx->s_comp));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->s_comp));
    return 0;
}

int b200h::hex_rows_from_host(b200h_ctx* ctx, const uint8_t* raw, uint64_t nbytes, uint8_t* out) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!nbytes) return 0;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t at = (nbytes + 255) & ~uint64_t(255);
    if (int rc = ensure_dev(ctx, ctx->d_hex, at + 2 * nbytes + 64)) return rc;
    uint8_t* d_raw = (uint8_t*)ctx->d_hex.p;
    CU_TRY(ctx, cudaMemcpyAsync(d_raw, raw, nbytes, cudaMemcpyHostToDevice, ctx->s_comp));
    ctx->launches += launch_hex_rows(d_raw, nbytes, d_raw + at, ctx->s_comp);
    CU_TRY(ctx, cudaGetLastError());
    CU_TRY(ctx, cudaMemcpyAsync(out, d_raw + at, 2 * nbytes, cudaMemcpyDefault, ctx->s_comp));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->s_comp));
    return 0;
}

extern "C" {

void b200h_destroy(b200h_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto& pr : ctx->prof_events) {
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    for (DevBuf* b : {&ctx->d_off, &ctx->d_len, &ctx->d_order, &ctx->d_trim, &ctx->d_sha, &ctx->d_md5, &ctx->d_scratch,
                      &ctx->d_small, &ctx->d_states, &ctx->d_dedupe, &ctx->d_keys, &ctx->d_trimctl, &ctx->d_hex, &ctx->d_order_long})
        if (b->p) cudaFree(b->p);
    for (auto& r : ctx->stream_pool) stream_res_destroy(r);
    ctx->stream_pool.clear();
    for (int s = 0; s < 2; ++s) {
        if (ctx->dwave[s]) cudaFree(ctx->dwave[s]);
        if (ctx->pin[s]) cudaFreeHost(ctx->pin[s]);
        if (ctx->ev_copied[s]) cudaEventDestroy(ctx->ev_copied[s]);
        if (ctx->ev_consumed[s]) cudaEventDestroy(ctx->ev_consumed[s]);
        if (ctx->ev_pin[s]) cudaEventDestroy(ctx->ev_pin[s]);
    }
    if (ctx->ev_scratch) cudaEventDestroy(ctx->ev_scratch);
    if (ctx->ev_dedupe) cudaEventDestroy(ctx->ev_dedupe);
    if (ctx->h_meta) cudaFreeHost(ctx->h_meta);
    if (ctx->h_plan) cudaFreeHost(ctx->h_plan);
    if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
    if (ctx->s_comp) cudaStreamDestroy(ctx->s_comp);
    if (ctx->s_chain) cudaStreamDestroy(ctx->s_chain);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    cudaGetLastError();
    delete ctx;
}

void* b200h_host_alloc(b200h_ctx* ctx, size_t bytes) {
    if (!ctx) return nullptr;
    std::lock_guard<std::mutex> lk(ctx->mu);
    void* p = nullptr;
    if (cudaSetDevice(ctx->device) != cudaSuccess || cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        ctx->err = std::string("cudaHostAlloc failed: ") + cudaGetErrorString(cudaGetLastError());
        return nullptr;
    }
    return p;
}

void b200h_host_free(b200h_ctx* ctx, void* p) {
    if (!ctx || !p) return;
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaFreeHost(p);
    cudaGetLastError();
}

int b200h_hash_batch_host(b200h_ctx* ctx, const uint8_t* base, const uint64_t* offsets, const uint64_t* lengths,
                          uint64_t n, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                          uint64_t* trimmed_len_out) {
    if (!ctx) return B200H_E_INVALID;
    B200H_RANGE("b200h_hash_batch_host");
    if (n && n <= kCombineMaxN && ctx->combine_enabled && offsets && lengths && (flags & (B200H_SHA256 | B200H_MD5)) &&
        !(flags & B200H_HEX_OUT))
        return combined_hash_batch_host(ctx, base, offsets, lengths, n, flags & kPublicFlags, sha256_out, md5_out,
                                        trimmed_len_out);
    std::lock_guard<std::mutex> lk(ctx->mu);
    return hash_batch_host_impl(ctx, base, offsets, lengths, n, flags & kPublicFlags, sha256_out, md5_out,
                                trimmed_len_out, nullptr);
}

int b200h_hash_batch_device_hl(b200h_ctx* ctx, const void* d_base, const uint64_t* d_offsets, const uint64_t* d_lengths,
                               const uint64_t* h_lengths, uint64_t n, uint32_t flags, void* d_sha256, void* d_md5,
                               uint64_t* d_trimmed_len, void* cuda_stream) {
    if (!ctx) return B200H_E_INVALID;
    B200H_RANGE("b200h_hash_batch_device");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (n && (!d_offsets || !d_lengths)) return fail(ctx, B200H_E_INVALID, "offsets/lengths must not be NULL");
    if (((uintptr_t)d_sha256 | (uintptr_t)d_md5) & 15u)
        return fail(ctx, B200H_E_INVALID, "digest outputs must be 16-byte aligned");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->s_comp;
    uint8_t* o_sha = (flags & B200H_SHA256) ? (uint8_t*)d_sha256 : nullptr;
    uint8_t* o_md5 = (flags & B200H_MD5) ? (uint8_t*)d_md5 : nullptr;
    if (!(flags & B200H_HEX_OUT) || !n)
        return enqueue_device_batch(ctx, (const uint8_t*)d_base, d_offsets, d_lengths, n, flags & kPublicFlags, o_sha, o_md5,
                                    d_trimmed_len, nullptr, st, h_lengths);
    // hex columns: the kernels write raw rows into library scratch, hex_rows_kernel expands them into the caller's
    // (twice as wide) buffers, all on `st`
    if (ctx->scratch_used) CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_scratch, 0));
    if (int rc = ensure_dev(ctx, ctx->d_hex, n * 48 + 64)) return rc;
    uint8_t* raw_sha = (uint8_t*)ctx->d_hex.p;
    uint8_t* raw_md5 = raw_sha + n * 32;
    if (int rc = enqueue_device_batch(ctx, (const uint8_t*)d_base, d_offsets, d_lengths, n, flags & kPublicFlags,
                                      o_sha ? raw_sha : nullptr, o_md5 ? raw_md5 : nullptr, d_trimmed_len, nullptr, st, h_lengths))
        return rc;
    if (o_sha) ctx->launches += launch_hex_rows(raw_sha, n * 32, o_sha, st);
    if (o_md5) ctx->launches += launch_hex_rows(raw_md5, n * 16, o_md5, st);
    CU_TRY(ctx, cudaGetLastError());
    CU_TRY(ctx, cudaEventRecord(ctx->ev_scratch, st));  // d_hex is shared scratch like the planner's
    return 0;
}

int b200h_hash_batch_device(b200h_ctx* ctx, const void* d_base, const uint64_t* d_offsets, const uint64_t* d_lengths,
                            uint64_t n, uint32_t flags, void* d_sha256, void* d_md5, uint64_t* d_trimmed_len,
                            void* cuda_stream) {
    return b200h_hash_batch_device_hl(ctx, d_base, d_offsets, d_lengths, nullptr, n, flags, d_sha256, d_md5,
                                      d_trimmed_len, cuda_stream);
}

int b200h_hash_fixed_parts(b200h_ctx* ctx, const uint8_t* base, uint64_t len, uint64_t part_len, uint32_t flags,
                           uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out, uint8_t etag_md5_out[16],
                           uint64_t* nparts_out) {
    if (!ctx) return B200H_E_INVALID;
    B200H_RANGE("b200h_hash_fixed_parts");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (part_len == 0) return fail(ctx, B200H_E_INVALID, "part_len must be > 0");
    const uint64_t nparts = (len + part_len - 1) / part_len;
    if (nparts_out) *nparts_out = nparts;
    if (nparts == 0) {
        if (etag_md5_out) {
            // md5 of the empty concatenation: hash one empty message
            uint64_t z = 0;
            return hash_batch_host_impl(ctx, base ? base : (const uint8_t*)&z, &z, &z, 1, B200H_MD5, nullptr,
                                        etag_md5_out, nullptr, nullptr);
        }
        return 0;
    }
    std::vector<uint64_t> off(nparts), ln(nparts);
    for (uint64_t i = 0; i < nparts; ++i) {
        off[i] = i * part_len;
        ln[i] = std::min(part_len, len - off[i]);
    }
    return hash_batch_host_impl(ctx, base, off.data(), ln.data(), nparts, flags & kPublicFlags, sha256_out, md5_out,
                                trimmed_len_out, etag_md5_out);
}

// ---------------------------------------------------------------------------------------------- files

int b200h_stat_files(b200h_ctx* ctx, const char* const* paths, uint64_t n, uint64_t* sizes_out, uint32_t* modes_out) {
    if (!ctx) return B200H_E_INVALID;
    B200H_RANGE("b200h_stat_files");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (n && (!paths || !sizes_out)) return fail(ctx, B200H_E_INVALID, "paths/sizes_out must not be NULL");
    std::atomic<int> err{0};
    std::atomic<uint64_t> bad{0};
    const int t = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)ctx->io_threads, n / 256));
    auto work = [&](uint64_t a, uint64_t b) {
        for (uint64_t i = a; i < b && !err.load(std::memory_order_relaxed); ++i) {
            struct stat sb;
            if (stat(paths[i], &sb) != 0 || !S_ISREG(sb.st_mode)) {
                int expected = 0;
                if (err.compare_exchange_strong(expected, errno ? errno : EINVAL)) bad.store(i);
                return;
            }
            sizes_out[i] = (uint64_t)sb.st_size;
            if (modes_out) modes_out[i] = (uint32_t)(sb.st_mode & 07777);
        }
    };
    if (t <= 1) {
        work(0, n);
    } else {
        std::vector<std::thread> th;
        for (int k = 0; k < t; ++k) th.emplace_back(work, n * k / t, n * (k + 1) / t);
        for (auto& x : th) x.join();
    }
    if (err.load()) return fail(ctx, B200H_E_IO, std::string("stat ") + paths[bad.load()] + ": " + strerror(err.load()));
    return 0;
}

int b200h_hash_files(b200h_ctx* ctx, const char* const* paths, uint64_t n, const uint64_t* sizes, uint64_t part_len,
                     uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out) {
    if (!ctx) return B200H_E_INVALID;
    B200H_RANGE("b200h_hash_files");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (n && (!paths || !sizes)) return fail(ctx, B200H_E_INVALID, "paths/sizes must not be NULL");
    std::vector<uint64_t> off, len, file_of;
    b200h::file_messages(sizes, n, part_len, off, len, file_of);
    if (off.empty()) return 0;
    return hash_batch_host_impl(ctx, nullptr, off.data(), len.data(), off.size(), flags & kPublicFlags, sha256_out,
                                md5_out, trimmed_len_out, nullptr, paths, file_of.data());
}

// ------------------------------------------------------------------------------------------ streaming
// A b200h_stream owns a CUDA stream, a pinned accumulation buffer and a device block that holds everything its
// launches touch (chaining state, planner scratch, queue ring, data), so several streams of one context -- the
// reference hashes files from ThreadPool / to_thread workers, one hashlib object each -- advance concurrently on the
// GPU, one chain per stream.  update() only copies into the pinned buffer; every `cap` bytes one absorb is enqueued
// (H2D + plan + chain kernel) and update() returns without waiting for it: the next absorb's bytes are gathered
// while the GPU works on this one.  The host knows every length, so nothing is read back.

extern "C++" {
namespace {

constexpr size_t kStreamStateBytes = 2 * sizeof(ChainState);  // [0] running, [1] scratch copy for digest()
constexpr size_t kStreamMetaOff = kStreamStateBytes;          // 2 x u64
constexpr size_t kStreamOutOff = kStreamMetaOff + 64;         // 32 + 16
constexpr size_t kStreamPlanOff = kStreamOutOff + 64;         // planner scratch + chain list
constexpr size_t kStreamPlanBytes = (kPlanScratchWords + kMaxChain) * sizeof(uint32_t);
constexpr size_t kStreamRingOff = (kStreamPlanOff + kStreamPlanBytes + 127) & ~size_t(127);
constexpr size_t kStreamRingBytes = 32 * sizeof(uint32_t);    // ring_capacity(1)
constexpr size_t kStreamDataOff = (kStreamRingOff + kStreamRingBytes + 255) & ~size_t(255);

int stream_res_acquire(b200h_ctx* ctx, b200h_ctx::StreamBuf* out) {
    if (!ctx->stream_pool.empty()) {
        *out = ctx->stream_pool.back();
        ctx->stream_pool.pop_back();
        return 0;
    }
    b200h_ctx::StreamBuf r;
    cudaError_t e = cudaHostAlloc(&r.h, ctx->stream_cap + 128, cudaHostAllocDefault);  // + pinned {offset, length} slots and digests
    if (e == cudaSuccess) e = cudaMalloc(&r.d, kStreamDataOff + ctx->stream_cap + 64);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r.st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r.ev, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (r.h) cudaFreeHost(r.h);
        if (r.d) cudaFree(r.d);
        if (r.st) cudaStreamDestroy(r.st);
        if (r.ev) cudaEventDestroy(r.ev);
        return fail(ctx, B200H_E_NOMEM, std::string("stream allocation failed: ") + cudaGetErrorString(e));
    }
    *out = r;
    return 0;
}

void stream_res_destroy(b200h_ctx::StreamBuf& r) {
    if (r.st) cudaStreamSynchronize(r.st);
    if (r.h) cudaFreeHost(r.h);
    if (r.d) cudaFree(r.d);
    if (r.st) cudaStreamDestroy(r.st);
    if (r.ev) cudaEventDestroy(r.ev);
    cudaGetLastError();
    r = b200h_ctx::StreamBuf();
}

int stream_write_iv(b200h_stream* s) {
    b200h_ctx* ctx = s->ctx;
    ChainState init;
    memcpy(init.sha, kShaIv, sizeof kShaIv);
    memcpy(init.md5, kMd5Iv, sizeof kMd5Iv);
    init.prior_bytes = 0;
    init.reserved = 0;
    // {0, cap}: offset and length of every absorb, device-resident for the life of the stream (no per-absorb copy)
    uint64_t* h_meta = reinterpret_cast<uint64_t*>(s->hbuf + s->cap);
    h_meta[0] = 0;
    h_meta[1] = s->cap;
    CU_TRY(ctx, cudaMemcpyAsync(s->d_state, &init, sizeof init, cudaMemcpyHostToDevice, s->res.st));
    CU_TRY(ctx, cudaMemcpyAsync(s->d_meta, h_meta, 2 * sizeof(uint64_t), cudaMemcpyHostToDevice, s->res.st));
    CU_TRY(ctx, cudaStreamSynchronize(s->res.st));  // also drains whatever the stream still had in flight
    s->h2d_pending = false;
    s->fill = 0;
    s->total = 0;
    return 0;
}

// hbuf may be rewritten once the last copy out of it has finished (waits outside the context lock)
int stream_wait_hbuf(b200h_stream* s) {
    if (s->h2d_pending) {
        CU_TRY(s->ctx, cudaEventSynchronize(s->res.ev));
        s->h2d_pending = false;
    }
    return 0;
}

// enqueue: absorb the first `nbytes` (multiple of 64) of hbuf into the running state.  ctx->mu must be held.
int stream_absorb(b200h_stream* s, size_t nbytes) {
    b200h_ctx* ctx = s->ctx;
    if (nbytes != s->cap) return fail(ctx, B200H_E_STATE, "stream absorbs whole buffers only");
    const uint64_t hlen = nbytes;
    cudaStream_t st = s->res.st;
    CU_TRY(ctx, cudaMemcpyAsync(s->d_buf, s->hbuf, nbytes, cudaMemcpyHostToDevice, st));  // pinned: truly asynchronous
    CU_TRY(ctx, cudaEventRecord(s->res.ev, st));
    s->h2d_pending = true;
    return enqueue_device_batch(ctx, s->d_buf, s->d_meta, s->d_meta + 1, 1, (s->flags & 3u) | kFlagNoFinal, nullptr,
                                nullptr, nullptr, s->d_state, st, &hlen, s->d_plan, s->d_ring);
}

}  // namespace
}  // extern "C++"

int b200h_stream_new(b200h_ctx* ctx, uint32_t flags, b200h_stream** out) {
    if (!ctx || !out) return B200H_E_INVALID;
    B200H_RANGE("b200h_stream_new");
    std::lock_guard<std::mutex> lk(ctx->mu);
    *out = nullptr;
    if (!(flags & (B200H_SHA256 | B200H_MD5))) return fail(ctx, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    b200h_stream* s = new (std::nothrow) b200h_stream();
    if (!s) return fail(ctx, B200H_E_NOMEM, "out of host memory");
    s->ctx = ctx;
    s->flags = flags & 3u;
    s->cap = ctx->stream_cap;
    if (int rc = stream_res_acquire(ctx, &s->res)) {
        delete s;
        return rc;
    }
    uint8_t* blk = s->res.d;
    s->hbuf = s->res.h;
    s->d_state = (ChainState*)blk;
    s->d_meta = (uint64_t*)(blk + kStreamMetaOff);
    s->d_out = blk + kStreamOutOff;
    s->d_plan = (uint32_t*)(blk + kStreamPlanOff);
    s->d_ring = (uint32_t*)(blk + kStreamRingOff);
    s->d_buf = blk + kStreamDataOff;
    if (int rc = stream_write_iv(s)) {
        stream_res_destroy(s->res);
        delete s;
        return rc;
    }
    *out = s;
    return 0;
}

int b200h_stream_update(b200h_stream* s, const uint8_t* data, uint64_t len) {
    if (!s) return B200H_E_INVALID;
    B200H_RANGE("b200h_stream_update");
    b200h_ctx* ctx = s->ctx;
    if (len && !data) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        return fail(ctx, B200H_E_INVALID, "data is NULL");
    }
    if (cudaSetDevice(ctx->device) != cudaSuccess) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        CU_TRY(ctx, cudaSetDevice(ctx->device));
    }
    s->total += len;
    while (len) {
        if (s->fill == 0)
            if (int rc = stream_wait_hbuf(s)) return rc;
        const size_t take = (size_t)std::min<uint64_t>(len, s->cap - s->fill);
        memcpy(s->hbuf + s->fill, data, take);
        s->fill += take;
        data += take;
        len -= take;
        if (s->fill == s->cap) {
            std::lock_guard<std::mutex> lk(ctx->mu);  // enqueue only: microseconds
            if (int rc = stream_absorb(s, s->cap)) return rc;
            s->fill = 0;
        }
    }
    return 0;
}

int b200h_stream_digest(b200h_stream* s, uint8_t sha256_out[32], uint8_t md5_out[16]) {
    if (!s) return B200H_E_INVALID;
    B200H_RANGE("b200h_stream_digest");
    b200h_ctx* ctx = s->ctx;
    cudaStream_t st = s->res.st;
    uint8_t* host = s->hbuf + s->cap + 64;  // pinned: the copy below only enqueues
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        CU_TRY(ctx, cudaSetDevice(ctx->device));
        // finalise on a scratch copy of the state so that further updates remain possible
        uint64_t* h_meta = reinterpret_cast<uint64_t*>(s->hbuf + s->cap) + 2;  // pinned slot of the digest launch
        h_meta[0] = 0;
        h_meta[1] = s->fill;
        const uint64_t hlen = s->fill;
        CU_TRY(ctx, cudaMemcpyAsync(s->d_state + 1, s->d_state, sizeof(ChainState), cudaMemcpyDeviceToDevice, st));
        if (s->fill) CU_TRY(ctx, cudaMemcpyAsync(s->d_buf, s->hbuf, s->fill, cudaMemcpyHostToDevice, st));
        CU_TRY(ctx, cudaMemcpyAsync(s->d_meta + 2, h_meta, 2 * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
        if (int rc = enqueue_device_batch(ctx, s->d_buf, s->d_meta + 2, s->d_meta + 3, 1, s->flags, s->d_out, s->d_out + 32,
                                          nullptr, s->d_state + 1, st, &hlen, s->d_plan, s->d_ring))
            return rc;
        CU_TRY(ctx, cudaMemcpyAsync(host, s->d_out, 48, cudaMemcpyDeviceToHost, st));
    }
    CU_TRY(ctx, cudaStreamSynchronize(st));  // outside the lock: other streams keep enqueueing meanwhile
    s->h2d_pending = false;
    if (sha256_out && (s->flags & B200H_SHA256)) memcpy(sha256_out, host, 32);
    if (md5_out && (s->flags & B200H_MD5)) memcpy(md5_out, host + 32, 16);
    return 0;
}

int b200h_stream_reset(b200h_stream* s) {
    if (!s) return B200H_E_INVALID;
    std::lock_guard<std::mutex> lk(s->ctx->mu);
    CU_TRY(s->ctx, cudaSetDevice(s->ctx->device));
    return stream_write_iv(s);
}

void b200h_stream_free(b200h_stream* s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->res.st);
    cudaGetLastError();
    {
        std::lock_guard<std::mutex> lk(s->ctx->mu);
        if (s->ctx->stream_pool.size() < 64) s->ctx->stream_pool.push_back(s->res);
        else stream_res_destroy(s->res);
    }
    delete s;
}

// ---- dedupe of the digest table ------------------------------------------------------------------

static int dedupe_args_ok(b200h_ctx* ctx, uint64_t n, uint32_t key_bytes) {
    if (!ctx) return B200H_E_INVALID;
    if (key_bytes != 32 && key_bytes != 16) return fail(ctx, B200H_E_INVALID, "key_bytes must be 32 (SHA-256) or 16 (MD5)");
    if (n >= 0x7fffffffull) return fail(ctx, B200H_E_INVALID, "table larger than 2^31-2 rows");
    return 0;
}

int b200h_dedupe_device(b200h_ctx* ctx, const void* d_keys, uint64_t n, uint32_t key_bytes, uint32_t* d_first,
                        uint64_t* d_ndistinct, void* cuda_stream) {
    if (int rc = dedupe_args_ok(ctx, n, key_bytes)) return rc;
    if (n && (!d_keys || !d_first)) return fail(ctx, B200H_E_INVALID, "null device pointer");
    if ((reinterpret_cast<uintptr_t>(d_keys) & 3) != 0) return fail(ctx, B200H_E_INVALID, "d_keys must be 4-byte aligned");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->s_comp;
    if (int rc = ensure_dev(ctx, ctx->d_dedupe, (size_t)dedupe_table_capacity(n) * 2 * sizeof(uint32_t))) return rc;
    if (ctx->dedupe_used) CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_dedupe, 0));  // table shared across streams
    ctx->launches += launch_dedupe(d_keys, n, key_bytes, (uint32_t*)ctx->d_dedupe.p, d_first,
                                   reinterpret_cast<unsigned long long*>(d_ndistinct), st);
    CU_TRY(ctx, cudaGetLastError());
    CU_TRY(ctx, cudaEventRecord(ctx->ev_dedupe, st));
    ctx->dedupe_used = true;
    return 0;
}

int b200h_dedupe_host(b200h_ctx* ctx, const uint8_t* keys, uint64_t n, uint32_t key_bytes, uint32_t* first_out,
                      uint64_t* ndistinct_out) {
    if (int rc = dedupe_args_ok(ctx, n, key_bytes)) return rc;
    if (n && (!keys || !first_out)) return fail(ctx, B200H_E_INVALID, "null pointer");
    if (n == 0) {
        if (ndistinct_out) *ndistinct_out = 0;
        return 0;
    }
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->s_comp;
    // device layout: keys | first[n] | ndistinct (8-byte aligned)
    const size_t kb = (size_t)n * key_bytes, fb = ((size_t)n * 4 + 7) & ~size_t(7);
    if (int rc = ensure_dev(ctx, ctx->d_keys, kb + fb + 8)) return rc;
    if (int rc = ensure_dev(ctx, ctx->d_dedupe, (size_t)dedupe_table_capacity(n) * 2 * sizeof(uint32_t))) return rc;
    uint8_t* d = (uint8_t*)ctx->d_keys.p;
    uint32_t* d_first = (uint32_t*)(d + kb);
    unsigned long long* d_cnt = (unsigned long long*)(d + kb + fb);
    if (ctx->dedupe_used) CU_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_dedupe, 0));
    CU_TRY(ctx, cudaMemcpyAsync(d, keys, kb, cudaMemcpyHostToDevice, st));
    ctx->launches += launch_dedupe(d, n, key_bytes, (uint32_t*)ctx->d_dedupe.p, d_first, d_cnt, st);
    CU_TRY(ctx, cudaGetLastError());
    CU_TRY(ctx, cudaMemcpyAsync(first_out, d_first, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    unsigned long long cnt = 0;
    CU_TRY(ctx, cudaMemcpyAsync(&cnt, d_cnt, 8, cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaStreamSynchronize(st));
    if (ndistinct_out) *ndistinct_out = cnt;
    return 0;
}

// ------------------------------------------------------------------------------------------ utilities

int b200h_fill_synth_device(b200h_ctx* ctx, void* d_dst, uint64_t nbytes, uint64_t seed, uint64_t start,
                            void* cuda_stream) {
    if (!ctx) return B200H_E_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (((uintptr_t)d_dst & 7u) || (start & 7u)) return fail(ctx, B200H_E_INVALID, "dst/start must be 8-byte aligned");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->s_comp;
    ctx->launches += launch_fill_synth((uint8_t*)d_dst, nbytes, seed, start, st);
    CU_TRY(ctx, cudaGetLastError());
    return 0;
}

int b200h_pack_preview(const uint8_t* base, const uint64_t* offsets, const uint64_t* lengths, uint64_t n, uint8_t* dst,
                       uint64_t dst_bytes, uint64_t slot_bytes, int threads, uint64_t* packed_offsets_out) {
    if ((!offsets || !lengths) && n) return B200H_E_INVALID;
    if (!dst || threads < 1 || slot_bytes < 4096) return B200H_E_INVALID;
    // the layout a staged wave gets in hash_batch_host_impl: every message at the next multiple of 16
    std::vector<uint64_t> doff(n ? n : 1);
    uint64_t used = 0;
    for (uint64_t i = 0; i < n; ++i) {
        doff[i] = used;
        used += (lengths[i] + 15) & ~15ull;
    }
    if (used > dst_bytes) return B200H_E_INVALID;
    Source src;
    src.base = base;
    src.off = offsets;
    // ... filled slot by slot, as the pinned ring is, by a team that outlives the call like a context's does (one per
    // calling thread here: a context's team is protected by the context mutex, this one by being thread-local)
    static thread_local PackTeam team;
    for (uint64_t lo = 0; lo < used; lo += slot_bytes)
        pack_parallel(team, threads, src, lengths, doff.data(), 0, n, lo, std::min(used, lo + slot_bytes), dst + lo);
    if (packed_offsets_out)
        for (uint64_t i = 0; i < n; ++i) packed_offsets_out[i] = doff[i];
    return 0;
}

int b200h_plan_preview(const uint64_t* lengths, uint64_t n, uint32_t flags, uint32_t sm_count, uint32_t* n_chain_out,
                       uint32_t* n_long_out) {
    if ((!lengths && n) || !sm_count || !(flags & (B200H_SHA256 | B200H_MD5)) || n >= 0x7fffffffull) return B200H_E_INVALID;
    // the same arguments enqueue_device_batch passes for a context on such a device with the default settings
    const uint32_t max_chain = (flags & B200H_NO_OUTLIERS) ? 0u : std::min<uint32_t>(sm_count * 4u, kMaxChain);
    const uint32_t long_cap = std::min<uint32_t>(sm_count * 4u * 32u, kLongRingCapacity);
    uint32_t n_long = 0;
    const uint32_t n_chain = plan_outliers_host(lengths, n, max_chain, sm_count, long_cap, plan_ratio8(flags & 3u), &n_long);
    if (n_chain_out) *n_chain_out = n_chain;
    if (n_long_out) *n_long_out = n_long;
    return 0;
}

int b200h_last_outlier_count(b200h_ctx* ctx, uint32_t* count_out) {
    if (!ctx || !count_out) return B200H_E_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    *count_out = ctx->last_outliers;
    return 0;
}

int b200h_combine_stats(b200h_ctx* ctx, uint64_t* groups_out, uint64_t* requests_out) {
    if (!ctx) return B200H_E_INVALID;
    std::lock_guard<std::mutex> lk(ctx->combiner.m);
    if (groups_out) *groups_out = ctx->combiner.groups;
    if (requests_out) *requests_out = ctx->combiner.requests;
    return 0;
}

uint64_t b200h_plan_sync_count(b200h_ctx* ctx) {
    if (!ctx) return 0;
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->plan_syncs;
}

uint64_t b200h_launch_count(b200h_ctx* ctx) {
    if (!ctx) return 0;
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->launches;
}

int b200h_profile_enable(b200h_ctx* ctx, int on) {
    if (!ctx) return B200H_E_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->profiling = on != 0;
    return 0;
}

int b200h_profile_read(b200h_ctx* ctx, double* ms, uint64_t* launches) {
    if (!ctx) return B200H_E_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    for (auto& pr : ctx->prof_events) {
        CU_TRY(ctx, cudaEventSynchronize(pr.second));
        float t = 0.f;
        CU_TRY(ctx, cudaEventElapsedTime(&t, pr.first, pr.second));
        ctx->prof_ms += t;
        ctx->prof_n += 1;
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    ctx->prof_events.clear();
    if (ms) *ms = ctx->prof_ms;
    if (launches) *launches = ctx->prof_n;
    ctx->prof_ms = 0.0;
    ctx->prof_n = 0;
    return 0;
}

}  // extern "C"
