// b200hash_group.cu -- device groups: one process hashes its batches on several GPUs (C ABI: include/b200hash.h).
//
// A group owns one context per listed device and one parked worker thread per member.  A batch is dealt over the
// members by bytes (split_owner), every worker hashes its member's share through that member's context, and the rows
// are scattered back to the caller's message indices: with memcpy for host outputs, with scatter_rows_kernel for
// device outputs.  A worker only ever touches its own member, so no thread holds two member mutexes at once and
// concurrent group calls cannot deadlock; the calling thread holds none while it waits.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b200hash.h"
#include "b200hash_internal.h"

namespace {

thread_local std::string g_group_create_error;

// dst[idx[r] * width + b] = src[r * width + b] for the `rows` rows of one member's share: raw or hex digest rows and
// 8-byte hashed lengths into the caller's table.  dst may be another device's memory reached over peer access.
__global__ void scatter_rows_kernel(const uint8_t* __restrict__ src, const uint64_t* __restrict__ idx, uint64_t rows,
                                    uint32_t width, uint8_t* __restrict__ dst) {
    const uint64_t total = rows * width;
    for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r = t / width;
        dst[idx[r] * width + (t - r * width)] = src[t];
    }
}

// A member's thread: started with the group, parked on a condition variable between jobs, joined in destroy.
class Worker {
public:
    Worker() : th_([this] { loop(); }) {}
    Worker(const Worker&) = delete;
    Worker& operator=(const Worker&) = delete;
    ~Worker() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
        }
        cv_.notify_one();
        th_.join();
    }
    void post(std::function<void()> job) {
        {
            std::lock_guard<std::mutex> lk(m_);
            q_.push_back(std::move(job));
        }
        cv_.notify_one();
    }

private:
    void loop() {
        for (;;) {
            std::function<void()> job;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
                if (q_.empty()) return;
                job = std::move(q_.front());
                q_.pop_front();
            }
            job();
        }
    }

    std::mutex m_;
    std::condition_variable cv_;
    std::deque<std::function<void()>> q_;
    bool stop_ = false;
    std::thread th_;  // last: the thread starts once the members above exist
};

struct DevScratch {
    int device = -1;
    uint8_t* p = nullptr;
    size_t cap = 0;
};

// Everything below `worker` is touched by the worker thread only.
struct Member {
    b200h_ctx* ctx = nullptr;
    int device = 0;
    std::unique_ptr<Worker> worker;
    cudaStream_t st = nullptr;          // on `device`
    DevScratch share;                   // on `device`: the share's device output columns, then its row indices
    DevScratch staged;                  // on the table device when it cannot reach `share` over peer access
    cudaStream_t st_table = nullptr;    // on staged.device
    std::vector<signed char> peer;      // per table device: -1 not asked yet, 0 no peer access, 1 enabled
};

// The output columns of a batch: sha256 | md5 | hashed length.
struct Columns {
    uint8_t* out[3] = {nullptr, nullptr, nullptr};
    uint32_t width[3] = {0, 0, 8};
    bool on_device[3] = {false, false, false};
    int table_device = -1;
};

struct Share {
    std::vector<uint64_t> idx, off, len, file_of;
    std::vector<uint64_t> piece_of{0}, psrc, plen;  // gathered rows of a device-segments share (b200h::GatherRows)
    uint64_t bytes = 0, staged = 0;
    double ms = 0.0;
    int rc = 0;
    std::string err;
};

}  // namespace

struct b200h_group {
    std::vector<std::unique_ptr<Member>> members;
    uint64_t min_share = B200H_GROUP_MIN_SHARE;
    std::mutex mu;  // err and the last split
    std::string err;
    std::vector<uint64_t> last_messages, last_bytes, last_staged;
    std::vector<double> last_ms;
};

namespace {

using Clock = std::chrono::steady_clock;

double ms_since(Clock::time_point t0) { return std::chrono::duration<double, std::milli>(Clock::now() - t0).count(); }

std::string cuda_msg(const char* what, cudaError_t e) {
    cudaGetLastError();
    return std::string(what) + " failed: " + cudaGetErrorString(e);
}

// k = min(members, n, max(1, total / min_share)); messages sorted by length (longest first, stable) and dealt over
// 0..k-1 in boustrophedon order -- the same deal as sharding.shard_assignment(lengths, k).
int split_owner(const uint64_t* len, uint64_t n, int nmembers, uint64_t min_share, uint32_t* owner) {
    if (min_share == 0) min_share = B200H_GROUP_MIN_SHARE;
    uint64_t total = 0;
    for (uint64_t i = 0; i < n; ++i) total += len[i];
    const uint64_t k = std::min<uint64_t>({(uint64_t)std::max(nmembers, 0), n, std::max<uint64_t>(1, total / min_share)});
    if (k == 0) return 0;
    std::vector<uint64_t> order(n);
    std::iota(order.begin(), order.end(), uint64_t(0));
    std::stable_sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return len[a] > len[b]; });
    for (uint64_t p = 0; p < n; ++p) {
        const uint64_t lap = p / k, col = p % k;
        owner[order[p]] = (uint32_t)((lap & 1) ? k - 1 - col : col);
    }
    return (int)k;
}

int group_fail(b200h_group* g, int code, const std::string& msg) {
    std::lock_guard<std::mutex> lk(g->mu);
    g->err = msg;
    return code;
}

std::string member_prefix(b200h_group* g, int j) {
    return "member " + std::to_string(j) + " (cuda:" + std::to_string(g->members[j]->device) + "): ";
}

// Host or device memory?  Device columns must all sit on one device.
int classify_outputs(b200h_group* g, Columns& c) {
    for (int k = 0; k < 3; ++k) {
        if (!c.out[k]) continue;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, c.out[k]) != cudaSuccess) {
            cudaGetLastError();
            continue;  // plain pageable host memory
        }
        if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) continue;
        if (c.table_device >= 0 && c.table_device != at.device)
            return group_fail(g, B200H_E_INVALID, "device outputs must all be on one device (got cuda:" +
                                                      std::to_string(c.table_device) + " and cuda:" +
                                                      std::to_string(at.device) + ")");
        c.on_device[k] = true;
        c.table_device = at.device;
    }
    return 0;
}

int ensure_scratch(DevScratch& s, int device, size_t bytes, std::string* err) {
    if (s.device == device && s.cap >= bytes) return 0;
    if (s.p) {
        cudaSetDevice(s.device);
        cudaFree(s.p);
        s.p = nullptr;
        s.cap = 0;
    }
    s.device = device;
    const size_t want = std::max<size_t>(bytes, size_t(1) << 20);
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s.p, want);
    if (e != cudaSuccess) {
        *err = cuda_msg("cudaMalloc (group scatter buffer)", e);
        s.p = nullptr;
        return e == cudaErrorMemoryAllocation ? B200H_E_NOMEM : B200H_E_CUDA;
    }
    s.cap = want;
    return 0;
}

// May the member's device write into memory on `table`?  Peer access is enabled for this process's contexts only.
bool peer_ok(Member& m, int table) {
    if (table == m.device) return true;
    if ((int)m.peer.size() <= table) m.peer.resize(table + 1, -1);
    if (m.peer[table] < 0) {
        int can = 0;
        m.peer[table] = 0;
        if (cudaDeviceCanAccessPeer(&can, m.device, table) == cudaSuccess && can) {
            cudaSetDevice(m.device);
            const cudaError_t e = cudaDeviceEnablePeerAccess(table, 0);
            m.peer[table] = (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) ? 1 : 0;
        }
        cudaGetLastError();
    }
    return m.peer[table] == 1;
}

int launch_scatter(const uint8_t* src, const uint64_t* idx, uint64_t rows, uint32_t width, uint8_t* dst, cudaStream_t st) {
    const uint64_t total = rows * width;
    const unsigned blocks = (unsigned)std::min<uint64_t>((total + 255) / 256, 148 * 16);
    scatter_rows_kernel<<<blocks, 256, 0, st>>>(src, idx, rows, width, dst);
    return 1;
}

#define GROUP_CU(call)                                   \
    do {                                                 \
        cudaError_t e__ = (call);                        \
        if (e__ != cudaSuccess) {                        \
            s.err = cuda_msg(#call, e__);                \
            return B200H_E_CUDA;                         \
        }                                                \
    } while (0)

// The device columns of a finished share (in m.share, column k at col_at[k], row indices at idx_at) into the table.
int scatter_device(Member& m, const Columns& c, Share& s, const size_t* col_at, size_t idx_at, size_t used) {
    const uint64_t rows = s.idx.size();
    if (!m.st) {
        GROUP_CU(cudaSetDevice(m.device));
        GROUP_CU(cudaStreamCreateWithFlags(&m.st, cudaStreamNonBlocking));
    }
    const uint8_t* from = m.share.p;
    int dev = m.device;
    cudaStream_t st = m.st;
    if (!peer_ok(m, c.table_device)) {
        // no peer access: move the share (columns and indices) to the table device and scatter there
        if (int rc = ensure_scratch(m.staged, c.table_device, used, &s.err)) return rc;
        if (m.st_table && m.staged.device != c.table_device) {
            cudaStreamDestroy(m.st_table);
            m.st_table = nullptr;
        }
        GROUP_CU(cudaSetDevice(c.table_device));
        if (!m.st_table) GROUP_CU(cudaStreamCreateWithFlags(&m.st_table, cudaStreamNonBlocking));
        GROUP_CU(cudaMemcpyPeerAsync(m.staged.p, c.table_device, m.share.p, m.device, idx_at, m.st_table));
        GROUP_CU(cudaMemcpyAsync(m.staged.p + idx_at, s.idx.data(), rows * 8, cudaMemcpyHostToDevice, m.st_table));
        from = m.staged.p;
        dev = c.table_device;
        st = m.st_table;
    } else {
        GROUP_CU(cudaSetDevice(dev));
        GROUP_CU(cudaMemcpyAsync(m.share.p + idx_at, s.idx.data(), rows * 8, cudaMemcpyHostToDevice, st));
    }
    for (int k = 0; k < 3; ++k)
        if (c.out[k] && c.on_device[k])
            launch_scatter(from + col_at[k], (const uint64_t*)(from + idx_at), rows, c.width[k], c.out[k], st);
    GROUP_CU(cudaGetLastError());
    GROUP_CU(cudaStreamSynchronize(st));
    return 0;
}

// What one worker does with its member's share: hash it into share-sized outputs, scatter the rows.  device_rows: the
// share's off[] are absolute addresses of parts resident on the member's device (b200h_group_hash_device_parts).
void run_share(b200h_group* g, int j, const uint8_t* base, const char* const* paths, uint32_t flags, const Columns& c,
               Share& s, bool device_rows = false) {
    const auto t0 = Clock::now();
    Member& m = *g->members[j];
    const uint64_t rows = s.idx.size();
    std::vector<uint8_t> host[3];
    uint8_t* to[3] = {nullptr, nullptr, nullptr};
    size_t col_at[3] = {0, 0, 0}, used = 0;
    for (int k = 0; k < 3; ++k) {
        if (!c.out[k]) continue;
        if (c.on_device[k]) {
            col_at[k] = used;
            used += (rows * c.width[k] + 255) & ~size_t(255);
        } else {
            host[k].resize(rows * c.width[k]);
            to[k] = host[k].data();
        }
    }
    const size_t idx_at = used;
    if (used) {
        used += rows * 8;
        if ((s.rc = ensure_scratch(m.share, m.device, used, &s.err))) return;
        for (int k = 0; k < 3; ++k)
            if (c.out[k] && c.on_device[k]) to[k] = m.share.p + col_at[k];
    }
    const b200h::GatherRows gr{s.piece_of.data(), s.psrc.data(), s.plen.data(), b200h::gather_cap()};
    if (device_rows)
        s.rc = b200h::hash_device_rows(m.ctx, s.off.data(), s.len.data(), rows, flags, to[0], to[1], (uint64_t*)to[2],
                                       nullptr, 0, nullptr, s.psrc.empty() ? nullptr : &gr);
    else
        s.rc = b200h::hash_share(m.ctx, base, s.off.data(), s.len.data(), rows, flags, to[0], to[1], (uint64_t*)to[2],
                                 paths, paths ? s.file_of.data() : nullptr, &s.staged);
    if (s.rc) {
        s.err = b200h_last_error(m.ctx);
    } else {
        for (int k = 0; k < 3; ++k) {
            if (!c.out[k] || c.on_device[k]) continue;
            const uint32_t w = c.width[k];
            for (uint64_t r = 0; r < rows; ++r) memcpy(c.out[k] + s.idx[r] * w, host[k].data() + r * w, w);
        }
        if (used) s.rc = scatter_device(m, c, s, col_at, idx_at, used);
    }
    s.ms = ms_since(t0);
}

void record_split(b200h_group* g, const std::vector<Share>& shares) {
    const size_t nm = g->members.size();
    g->last_messages.assign(nm, 0);
    g->last_bytes.assign(nm, 0);
    g->last_staged.assign(nm, 0);
    g->last_ms.assign(nm, 0.0);
    for (size_t j = 0; j < shares.size(); ++j) {
        g->last_messages[j] = shares[j].idx.size();
        g->last_bytes[j] = shares[j].bytes;
        g->last_staged[j] = shares[j].staged;
        g->last_ms[j] = shares[j].ms;
    }
}

// Deal messages (off, len, file_of) over the members (owner[i] = member of message i), run every non-empty share on
// its member's worker, wait for all of them.  gather: the pieces of device rows that are gathered before hashing.
int run_split(b200h_group* g, const uint8_t* base, const char* const* paths, const uint64_t* off, const uint64_t* len,
              const uint64_t* file_of, uint64_t n, uint32_t flags, const Columns& c, const uint32_t* owner,
              bool device_rows = false, const b200h::SegmentRows* gather = nullptr) {
    const int nm = (int)g->members.size();
    std::vector<Share> shares(nm);
    for (uint64_t i = 0; i < n; ++i) {
        Share& s = shares[owner[i]];
        s.idx.push_back(i);
        s.off.push_back(off[i]);
        s.len.push_back(len[i]);
        if (file_of) s.file_of.push_back(file_of[i]);
        if (gather) {
            for (uint64_t p = gather->piece_of[i]; p < gather->piece_of[i + 1]; ++p) {
                s.psrc.push_back(gather->psrc[p]);
                s.plen.push_back(gather->plen[p]);
            }
            s.piece_of.push_back(s.psrc.size());
        }
        s.bytes += len[i];
    }
    std::mutex dm;
    std::condition_variable dcv;
    int left = 0;
    for (int j = 0; j < nm; ++j) left += !shares[j].idx.empty();
    for (int j = 0; j < nm; ++j)
        if (!shares[j].idx.empty())
            g->members[j]->worker->post([&, j] {
                run_share(g, j, base, paths, flags, c, shares[j], device_rows);
                std::lock_guard<std::mutex> lk(dm);  // notify under the lock: the waiter's cv lives on its stack
                --left;
                dcv.notify_one();
            });
    {
        std::unique_lock<std::mutex> lk(dm);
        dcv.wait(lk, [&] { return left == 0; });
    }
    std::lock_guard<std::mutex> lk(g->mu);
    record_split(g, shares);
    for (int j = 0; j < nm; ++j)
        if (shares[j].rc) {
            g->err = member_prefix(g, j) + shares[j].err;
            return shares[j].rc;
        }
    return 0;
}

// k <= 1: the home member's own entry point, exactly (or member j's, when the one member a batch uses is not home).
template <typename F>
int run_home(b200h_group* g, uint64_t n, const uint64_t* len, F call, int j = 0) {
    b200h_ctx* home = g->members[j]->ctx;
    const auto t0 = Clock::now();
    const uint64_t staged0 = b200h::staged_bytes(home);
    const int rc = call(home);
    std::vector<Share> one(j + 1);
    one[j].idx.resize(n);
    for (uint64_t i = 0; i < n; ++i) one[j].bytes += len[i];
    one[j].staged = b200h::staged_bytes(home) - staged0;
    one[j].ms = ms_since(t0);
    std::lock_guard<std::mutex> lk(g->mu);
    record_split(g, one);
    if (rc) g->err = member_prefix(g, j) + b200h_last_error(home);
    return rc;
}

// The raw columns of a device-parts batch (hashed into host memory because ETags were asked for) into the caller's
// outputs: copied as they are, or formatted as hex on the home member's device.
int deliver_raw(b200h_group* g, const uint8_t* raw, uint64_t nbytes, uint8_t* out, bool hex) {
    if (!out || !nbytes) return 0;
    if (hex) {
        b200h_ctx* home = g->members[0]->ctx;
        if (int rc = b200h::hex_rows_from_host(home, raw, nbytes, out))
            return group_fail(g, rc, member_prefix(g, 0) + b200h_last_error(home));
        return 0;
    }
    const cudaError_t e = cudaMemcpy(out, raw, nbytes, cudaMemcpyDefault);
    if (e != cudaSuccess) return group_fail(g, B200H_E_CUDA, cuda_msg("cudaMemcpy (group outputs)", e));
    return 0;
}

// The group batch of device-resident rows (b200h_group_hash_device_parts / _segments): file b's rows
// [row_of[b], row_of[b + 1]) are on device buf_dev[b]; the rows on device d are dealt over the members on d.  gather
// (may be NULL): the pieces of the rows that must be gathered first.  one_member(ctx) = the whole call on one member.
template <typename F>
int group_device_rows(b200h_group* g, const std::vector<int>& buf_dev, uint64_t n, const std::vector<uint64_t>& addr,
                      const std::vector<uint64_t>& len, const std::vector<uint64_t>& row_of, const b200h::SegmentRows* gather,
                      uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out,
                      uint8_t* etag_md5_out, F one_member) {
    const int nm = (int)g->members.size();
    const uint64_t rows = addr.size();
    // the parts resident on device d are dealt over the members on d by the rule of every other group batch
    std::vector<uint32_t> owner(rows);
    std::vector<int> used;
    std::vector<int> devs(buf_dev.begin(), buf_dev.end());
    std::sort(devs.begin(), devs.end());
    devs.erase(std::unique(devs.begin(), devs.end()), devs.end());
    for (int d : devs) {
        std::vector<uint64_t> idx, dlen;
        for (uint64_t b = 0; b < n; ++b)
            if (buf_dev[b] == d)
                for (uint64_t r = row_of[b]; r < row_of[b + 1]; ++r) {
                    idx.push_back(r);
                    dlen.push_back(len[r]);
                }
        if (idx.empty()) continue;
        std::vector<int> on_d;
        for (int j = 0; j < nm; ++j)
            if (g->members[j]->device == d) on_d.push_back(j);
        std::vector<uint32_t> local(idx.size());
        const int k = split_owner(dlen.data(), idx.size(), (int)on_d.size(), g->min_share, local.data());
        for (size_t p = 0; p < idx.size(); ++p) owner[idx[p]] = (uint32_t)on_d[local[p]];
        for (int q = 0; q < k; ++q) used.push_back(on_d[q]);
    }
    if (used.size() <= 1) return run_home(g, rows, len.data(), one_member, used.empty() ? 0 : used[0]);
    const uint32_t wide = (flags & B200H_HEX_OUT) ? 2 : 1;
    Columns c;
    if (!etag_md5_out) {
        c.out[0] = (flags & B200H_SHA256) ? sha256_out : nullptr;
        c.out[1] = (flags & B200H_MD5) ? md5_out : nullptr;
        c.out[2] = (uint8_t*)trimmed_len_out;
        c.width[0] = 32 * wide;
        c.width[1] = 16 * wide;
        if (int rc = classify_outputs(g, c)) return rc;
        return run_split(g, nullptr, nullptr, addr.data(), len.data(), nullptr, rows, flags, c, owner.data(), true, gather);
    }
    // ETags need every raw MD5 row in one place: the shares land in host tables, the ETags are one batch over
    // segments of the MD5 table on the home member, then the columns go where the caller wants them.
    std::vector<uint8_t> tsha((flags & B200H_SHA256) ? rows * 32 : 0), tmd5(rows * 16 + 16);
    std::vector<uint64_t> ttrim(rows);
    c.out[0] = tsha.empty() ? nullptr : tsha.data();
    c.out[1] = tmd5.data();
    c.out[2] = (uint8_t*)ttrim.data();
    c.width[0] = 32;
    c.width[1] = 16;
    if (int rc = run_split(g, nullptr, nullptr, addr.data(), len.data(), nullptr, rows, flags & ~B200H_HEX_OUT, c,
                           owner.data(), true, gather))
        return rc;
    std::vector<uint64_t> eoff(n), elen(n);
    for (uint64_t b = 0; b < n; ++b) {
        eoff[b] = 16 * row_of[b];
        elen[b] = 16 * (row_of[b + 1] - row_of[b]);
    }
    b200h_ctx* home = g->members[0]->ctx;
    uint64_t staged = 0;
    if (int rc = b200h::hash_share(home, tmd5.data(), eoff.data(), elen.data(), n, B200H_MD5, nullptr, etag_md5_out,
                                   nullptr, nullptr, nullptr, &staged))
        return group_fail(g, rc, member_prefix(g, 0) + b200h_last_error(home));
    const bool hex = (flags & B200H_HEX_OUT) != 0;
    if (int rc = deliver_raw(g, tsha.data(), tsha.size(), sha256_out, hex)) return rc;
    if (int rc = deliver_raw(g, tmd5.data(), rows * 16, md5_out, hex)) return rc;
    return deliver_raw(g, (const uint8_t*)ttrim.data(), rows * 8, (uint8_t*)trimmed_len_out, false);
}

}  // namespace

extern "C" {

int b200h_group_create(const int* devices, int ndevices, size_t pinned_bytes, size_t device_bytes,
                       uint64_t min_share_bytes, b200h_group** out) {
    if (!out) {
        g_group_create_error = "out is NULL";
        return B200H_E_INVALID;
    }
    *out = nullptr;
    if (!devices || ndevices < 1) {
        g_group_create_error = "a group needs at least one device";
        return B200H_E_INVALID;
    }
    b200h_group* g = new (std::nothrow) b200h_group();
    if (!g) {
        g_group_create_error = "out of host memory";
        return B200H_E_NOMEM;
    }
    g->min_share = min_share_bytes ? min_share_bytes : B200H_GROUP_MIN_SHARE;
    for (int i = 0; i < ndevices; ++i) {
        b200h_ctx* ctx = nullptr;
        const int rc = b200h::create_member(devices[i], pinned_bytes, device_bytes, devices, ndevices, &ctx);
        if (rc) {
            g_group_create_error = "member " + std::to_string(i) + " (cuda:" + std::to_string(devices[i]) +
                                   "): " + b200h_last_error(nullptr);
            b200h_group_destroy(g);
            return rc;
        }
        std::unique_ptr<Member> m(new Member());
        m->ctx = ctx;
        m->device = devices[i];
        m->worker.reset(new Worker());
        g->members.push_back(std::move(m));
    }
    *out = g;
    return 0;
}

void b200h_group_destroy(b200h_group* g) {
    if (!g) return;
    for (auto& m : g->members) m->worker.reset();  // joins: no share is in flight after this
    for (auto& m : g->members) {
        for (DevScratch* s : {&m->share, &m->staged})
            if (s->p) {
                cudaSetDevice(s->device);
                cudaFree(s->p);
            }
        if (m->st) {
            cudaSetDevice(m->device);
            cudaStreamDestroy(m->st);
        }
        if (m->st_table) {
            cudaSetDevice(m->staged.device);
            cudaStreamDestroy(m->st_table);
        }
        b200h_destroy(m->ctx);
    }
    cudaGetLastError();
    delete g;
}

const char* b200h_group_last_error(b200h_group* g) { return g ? g->err.c_str() : g_group_create_error.c_str(); }

int b200h_group_size(b200h_group* g) { return g ? (int)g->members.size() : 0; }

b200h_ctx* b200h_group_member(b200h_group* g, int i) {
    if (!g || i < 0 || i >= (int)g->members.size()) return nullptr;
    return g->members[i]->ctx;
}

int b200h_group_hash_batch_host(b200h_group* g, const uint8_t* base, const uint64_t* offsets, const uint64_t* lengths,
                                uint64_t n, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                                uint64_t* trimmed_len_out) {
    if (!g) return B200H_E_INVALID;
    if (n && (!offsets || !lengths)) return group_fail(g, B200H_E_INVALID, "offsets/lengths must not be NULL");
    if (!(flags & (B200H_SHA256 | B200H_MD5))) return group_fail(g, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    std::vector<uint32_t> owner(n);
    const int k = n ? split_owner(lengths, n, (int)g->members.size(), g->min_share, owner.data()) : 0;
    if (k <= 1)
        return run_home(g, n, lengths, [&](b200h_ctx* home) {
            return b200h_hash_batch_host(home, base, offsets, lengths, n, flags, sha256_out, md5_out, trimmed_len_out);
        });
    const uint32_t wide = (flags & B200H_HEX_OUT) ? 2 : 1;
    Columns c;
    c.out[0] = (flags & B200H_SHA256) ? sha256_out : nullptr;
    c.out[1] = (flags & B200H_MD5) ? md5_out : nullptr;
    c.out[2] = (uint8_t*)trimmed_len_out;
    c.width[0] = 32 * wide;
    c.width[1] = 16 * wide;
    if (int rc = classify_outputs(g, c)) return rc;
    return run_split(g, base, nullptr, offsets, lengths, nullptr, n, flags, c, owner.data());
}

int b200h_group_hash_files(b200h_group* g, const char* const* paths, uint64_t n, const uint64_t* sizes,
                           uint64_t part_len, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                           uint64_t* trimmed_len_out) {
    if (!g) return B200H_E_INVALID;
    if (n && (!paths || !sizes)) return group_fail(g, B200H_E_INVALID, "paths/sizes must not be NULL");
    if (!(flags & (B200H_SHA256 | B200H_MD5))) return group_fail(g, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    std::vector<uint64_t> off, len, file_of;
    b200h::file_messages(sizes, n, part_len, off, len, file_of);
    const uint64_t rows = off.size();
    std::vector<uint32_t> owner(rows);
    const int k = rows ? split_owner(len.data(), rows, (int)g->members.size(), g->min_share, owner.data()) : 0;
    if (k <= 1)
        return run_home(g, rows, len.data(), [&](b200h_ctx* home) {
            return b200h_hash_files(home, paths, n, sizes, part_len, flags, sha256_out, md5_out, trimmed_len_out);
        });
    const uint32_t wide = (flags & B200H_HEX_OUT) ? 2 : 1;
    Columns c;
    c.out[0] = (flags & B200H_SHA256) ? sha256_out : nullptr;
    c.out[1] = (flags & B200H_MD5) ? md5_out : nullptr;
    c.out[2] = (uint8_t*)trimmed_len_out;
    c.width[0] = 32 * wide;
    c.width[1] = 16 * wide;
    if (int rc = classify_outputs(g, c)) return rc;
    return run_split(g, nullptr, paths, off.data(), len.data(), file_of.data(), rows, flags, c, owner.data());
}

int b200h_group_hash_device_parts(b200h_group* g, const void* const* d_bufs, const uint64_t* sizes, uint64_t n,
                                  uint64_t part_len, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                                  uint64_t* trimmed_len_out, uint8_t* etag_md5_out) {
    if (!g) return B200H_E_INVALID;
    if (n && (!d_bufs || !sizes)) return group_fail(g, B200H_E_INVALID, "d_bufs/sizes must not be NULL");
    if (!(flags & (B200H_SHA256 | B200H_MD5))) return group_fail(g, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    if (etag_md5_out && !(flags & B200H_MD5)) return group_fail(g, B200H_E_INVALID, "etag requires B200H_MD5");
    const int nm = (int)g->members.size();
    // where every buffer lives; a buffer may only be hashed by the members on its device
    std::vector<int> buf_dev(n);
    for (uint64_t i = 0; i < n; ++i) {
        std::string what;
        const int d = b200h::buffer_device(d_bufs[i], sizes[i], &what);
        if (d == -1) return group_fail(g, B200H_E_INVALID, "buffer " + std::to_string(i) + " is " + what);
        bool covered = d < 0;
        for (int j = 0; j < nm && !covered; ++j) covered = g->members[j]->device == d;
        if (!covered)
            return group_fail(g, B200H_E_INVALID, "buffer " + std::to_string(i) + " is on cuda:" + std::to_string(d) +
                                                      ", which is not in the group");
        buf_dev[i] = d >= 0 ? d : g->members[0]->device;  // an empty buffer reads nothing: the home device takes it
    }
    std::vector<uint64_t> addr, len, row_of;
    b200h::device_part_rows(d_bufs, sizes, n, part_len, addr, len, row_of);
    return group_device_rows(g, buf_dev, n, addr, len, row_of, nullptr, flags, sha256_out, md5_out, trimmed_len_out,
                             etag_md5_out, [&](b200h_ctx* m) {
                                 return b200h_hash_device_parts(m, d_bufs, sizes, n, part_len, flags, sha256_out, md5_out,
                                                                trimmed_len_out, etag_md5_out);
                             });
}

int b200h_group_hash_device_segments(b200h_group* g, const void* const* d_segs, const uint64_t* seg_sizes,
                                     const uint64_t* seg_of, uint64_t n_files, uint64_t part_len, uint32_t flags,
                                     uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out,
                                     uint8_t* etag_md5_out) {
    if (!g) return B200H_E_INVALID;
    const std::string bad = b200h::segment_args_error(d_segs, seg_sizes, seg_of, n_files);
    if (!bad.empty()) return group_fail(g, B200H_E_INVALID, bad);
    if (!(flags & (B200H_SHA256 | B200H_MD5))) return group_fail(g, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    if (etag_md5_out && !(flags & B200H_MD5)) return group_fail(g, B200H_E_INVALID, "etag requires B200H_MD5");
    const int nm = (int)g->members.size();
    // where every file lives; a file may only be hashed by the members on its device
    std::vector<int> file_dev;
    std::string err;
    if (b200h::segment_devices(d_segs, seg_sizes, seg_of, n_files, file_dev, &err)) return group_fail(g, B200H_E_INVALID, err);
    for (uint64_t i = 0; i < n_files; ++i) {
        const int d = file_dev[i];
        bool covered = d < 0;
        for (int j = 0; j < nm && !covered; ++j) covered = g->members[j]->device == d;
        if (!covered)
            return group_fail(g, B200H_E_INVALID, "file " + std::to_string(i) + " is on cuda:" + std::to_string(d) +
                                                      ", which is not in the group");
        if (d < 0) file_dev[i] = g->members[0]->device;  // an empty file reads nothing: the home device takes it
    }
    b200h::SegmentRows sr;
    b200h::segment_rows(d_segs, seg_sizes, seg_of, n_files, part_len, sr);
    return group_device_rows(g, file_dev, n_files, sr.addr, sr.len, sr.row_of, &sr, flags, sha256_out, md5_out,
                             trimmed_len_out, etag_md5_out, [&](b200h_ctx* m) {
                                 return b200h_hash_device_segments(m, d_segs, seg_sizes, seg_of, n_files, part_len, flags,
                                                                   sha256_out, md5_out, trimmed_len_out, etag_md5_out);
                             });
}

int b200h_group_last_split(b200h_group* g, uint64_t* messages_out, uint64_t* bytes_out, uint64_t* staged_bytes_out,
                           double* busy_ms_out) {
    if (!g) return B200H_E_INVALID;
    std::lock_guard<std::mutex> lk(g->mu);
    const size_t nm = g->members.size();
    for (size_t j = 0; j < nm; ++j) {
        const bool have = j < g->last_messages.size();
        if (messages_out) messages_out[j] = have ? g->last_messages[j] : 0;
        if (bytes_out) bytes_out[j] = have ? g->last_bytes[j] : 0;
        if (staged_bytes_out) staged_bytes_out[j] = have ? g->last_staged[j] : 0;
        if (busy_ms_out) busy_ms_out[j] = have ? g->last_ms[j] : 0.0;
    }
    return 0;
}

int b200h_group_split_preview(const uint64_t* lengths, uint64_t n, int nmembers, uint64_t min_share_bytes,
                              uint32_t* owner_out, int* members_used_out) {
    if ((n && (!lengths || !owner_out)) || nmembers < 1) return B200H_E_INVALID;
    const int k = n ? split_owner(lengths, n, nmembers, min_share_bytes, owner_out) : 0;
    if (members_used_out) *members_used_out = k;
    return 0;
}

}  // extern "C"
