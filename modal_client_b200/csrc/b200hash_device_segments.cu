// b200hash_device_segments.cu -- b200h_hash_device_segments: files made of device segments (a safetensors file is a
// header plus N tensors back to back), hashed as if each file were one buffer (C ABI: include/b200hash.h).
//
// The row table is built here on the host.  A part whose bytes lie in one segment is hashed in place (an absolute
// address into that segment); a part that straddles a segment boundary is a gathered row: its pieces are copied into
// a scratch buffer on the context's device by gather_pieces_kernel, in one launch per window, and every row -- in
// place and gathered -- goes to the context's trim -> plan -> lane/chain kernels in one batch (hash_device_rows in
// b200hash_api.cu).  The group form is b200h_group_hash_device_segments (b200hash_group.cu).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/b200hash.h"
#include "b200hash_internal.h"

namespace {

// Largest piece one warp copies; longer pieces are split into items of this size on the host, tiny ones stay whole.
constexpr uint64_t kGatherItem = 64ull << 10;
constexpr uint64_t kDefaultGatherBytes = 4ull << 30;

// One warp copies [src, src + len) to dst with V-wide loads and stores; V divides (src - dst) mod 16, so once dst is
// V-aligned so is src.  The head (up to dst's alignment) and the tail (< V bytes) go byte by byte.
template <typename V>
__device__ __forceinline__ void warp_copy(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, uint64_t len,
                                          unsigned lane) {
    constexpr uint64_t W = sizeof(V);
    uint64_t head = (W - ((uintptr_t)dst & (W - 1))) & (W - 1);
    if (head > len) head = len;
    if (lane < head) dst[lane] = src[lane];
    const uint64_t nv = (len - head) / W;
    const V* s = reinterpret_cast<const V*>(src + head);
    V* d = reinterpret_cast<V*>(dst + head);
#pragma unroll 4
    for (uint64_t i = lane; i < nv; i += 32) d[i] = __ldg(s + i);
    const uint64_t done = head + nv * W;
    if (done + lane < len) dst[done + lane] = src[done + lane];
}

// Item t of a window: copy len[t] bytes from src[t] to dst[t] (absolute device addresses).  One warp per item, warps
// striding over the items: a window holds a few 64 KiB items per straddling 8 MiB block and, for a state dict of
// small tensors, thousands of pieces of a few bytes each.
__global__ void __launch_bounds__(256) gather_pieces_kernel(const uint64_t* __restrict__ src,
                                                            const uint64_t* __restrict__ dst,
                                                            const uint64_t* __restrict__ len, uint64_t items) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t t = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < items; t += warps) {
        const uint8_t* s = reinterpret_cast<const uint8_t*>(src[t]);
        uint8_t* d = reinterpret_cast<uint8_t*>(dst[t]);
        const uint64_t n = len[t];
        const unsigned mis = (unsigned)(((uintptr_t)s ^ (uintptr_t)d) & 15);
        if (mis == 0)
            warp_copy<uint4>(s, d, n, lane);
        else if ((mis & 7) == 0)
            warp_copy<uint2>(s, d, n, lane);
        else if ((mis & 3) == 0)
            warp_copy<uint32_t>(s, d, n, lane);
        else if ((mis & 1) == 0)
            warp_copy<uint16_t>(s, d, n, lane);
        else
            warp_copy<uint8_t>(s, d, n, lane);
    }
}

}  // namespace

int b200h::launch_gather(const uint64_t* d_src, const uint64_t* d_dst, const uint64_t* d_len, uint64_t items,
                         cudaStream_t st) {
    if (!items) return 0;
    const unsigned blocks = (unsigned)std::min<uint64_t>((items + 7) / 8, 148 * 8);
    gather_pieces_kernel<<<blocks, 256, 0, st>>>(d_src, d_dst, d_len, items);
    return 1;
}

uint64_t b200h::gather_item_bytes() { return kGatherItem; }

uint64_t b200h::gather_cap() {
    if (const char* e = getenv("B200H_GATHER_BYTES")) {
        const unsigned long long v = strtoull(e, nullptr, 10);
        if (v) return v;
    }
    return kDefaultGatherBytes;
}

void b200h::segment_rows(const void* const* d_segs, const uint64_t* seg_sizes, const uint64_t* seg_of, uint64_t n_files,
                         uint64_t part_len, SegmentRows& o) {
    std::vector<uint64_t> sizes(n_files, 0), off, file_of;
    for (uint64_t i = 0; i < n_files; ++i)
        for (uint64_t s = seg_of[i]; s < seg_of[i + 1]; ++s) sizes[i] += seg_sizes[s];
    b200h::file_messages(sizes.data(), n_files, part_len, off, o.len, file_of);
    const uint64_t rows = off.size();
    o.addr.assign(rows, 0);
    o.seg.assign(rows, 0);
    o.seg_off.assign(rows, 0);
    o.piece_of.assign(1, 0);
    o.psrc.clear();
    o.plen.clear();
    o.row_of.assign(n_files + 1, 0);
    for (uint64_t r = 0; r < rows; ++r) o.row_of[file_of[r] + 1] += 1;
    for (uint64_t i = 0; i < n_files; ++i) o.row_of[i + 1] += o.row_of[i];
    auto base = [&](uint64_t s) { return d_segs ? (uint64_t)(uintptr_t)d_segs[s] : 0; };
    for (uint64_t i = 0; i < n_files; ++i) {
        uint64_t s = seg_of[i], s_start = 0;  // first segment that may hold the next row, and its file offset
        for (uint64_t r = o.row_of[i]; r < o.row_of[i + 1]; ++r) {
            const uint64_t at = off[r], end = at + o.len[r];
            if (o.len[r] == 0) {  // an empty file's one row reads nothing
                o.seg[r] = seg_of[i];
                o.piece_of.push_back(o.psrc.size());
                continue;
            }
            // zero-size segments are not boundaries: skip them with every segment that ends at or before the row
            while (seg_sizes[s] == 0 || s_start + seg_sizes[s] <= at) s_start += seg_sizes[s++];
            if (s_start + seg_sizes[s] >= end) {
                o.seg[r] = s;
                o.seg_off[r] = at - s_start;
                o.addr[r] = base(s) + (at - s_start);
            } else {
                for (uint64_t t = s, t_start = s_start; t_start < end; t_start += seg_sizes[t++]) {
                    if (seg_sizes[t] == 0) continue;
                    const uint64_t lo = std::max(at, t_start), hi = std::min(end, t_start + seg_sizes[t]);
                    o.psrc.push_back(base(t) + (lo - t_start));
                    o.plen.push_back(hi - lo);
                }
            }
            o.piece_of.push_back(o.psrc.size());
        }
    }
}

void b200h::gather_windows(const uint64_t* len, const uint64_t* piece_of, uint64_t rows, uint64_t window_bytes,
                           std::vector<uint64_t>& win, std::vector<uint64_t>& dst, std::vector<uint64_t>& win_bytes) {
    win.assign(1, 0);
    win_bytes.assign(1, 0);
    dst.assign(rows, 0);
    bool any = false;  // the current window holds a gathered row
    for (uint64_t r = 0; r < rows; ++r) {
        if (piece_of[r + 1] == piece_of[r]) continue;
        const uint64_t p = (len[r] + 15) & ~uint64_t(15);
        if (any && win_bytes.back() + p > window_bytes) {
            win.push_back(r);
            win_bytes.push_back(0);
        }
        dst[r] = win_bytes.back();
        win_bytes.back() += p;
        any = true;
    }
    win.push_back(rows);
}

int b200h::segment_devices(const void* const* d_segs, const uint64_t* seg_sizes, const uint64_t* seg_of,
                           uint64_t n_files, std::vector<int>& file_dev, std::string* err) {
    file_dev.assign(n_files, -2);
    for (uint64_t i = 0; i < n_files; ++i)
        for (uint64_t s = seg_of[i]; s < seg_of[i + 1]; ++s) {
            std::string what;
            const int d = b200h::buffer_device(d_segs[s], seg_sizes[s], &what);
            if (d == -2) continue;
            if (d == -1) {
                *err = "file " + std::to_string(i) + " segment " + std::to_string(s) + " is " + what;
                return -1;
            }
            if (file_dev[i] >= 0 && file_dev[i] != d) {
                *err = "file " + std::to_string(i) + " has segments on cuda:" + std::to_string(file_dev[i]) +
                       " and cuda:" + std::to_string(d);
                return -1;
            }
            file_dev[i] = d;
        }
    return 0;
}

std::string b200h::segment_args_error(const void* const* d_segs, const uint64_t* seg_sizes, const uint64_t* seg_of,
                                      uint64_t n_files) {
    if (n_files && !seg_of) return "seg_of must not be NULL";
    for (uint64_t i = 0; i < n_files; ++i)
        if (seg_of[i] > seg_of[i + 1]) return "seg_of must not decrease (file " + std::to_string(i) + ")";
    if (n_files && seg_of[n_files] > seg_of[0] && (!d_segs || !seg_sizes)) return "d_segs/seg_sizes must not be NULL";
    return "";
}

extern "C" {

int b200h_hash_device_segments(b200h_ctx* ctx, const void* const* d_segs, const uint64_t* seg_sizes,
                               const uint64_t* seg_of, uint64_t n_files, uint64_t part_len, uint32_t flags,
                               uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out, uint8_t* etag_md5_out) {
    if (!ctx) return B200H_E_INVALID;
    const std::string bad = b200h::segment_args_error(d_segs, seg_sizes, seg_of, n_files);
    if (!bad.empty()) return b200h::ctx_fail(ctx, B200H_E_INVALID, bad);
    if (!(flags & (B200H_SHA256 | B200H_MD5)))
        return b200h::ctx_fail(ctx, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    if (etag_md5_out && !(flags & B200H_MD5)) return b200h::ctx_fail(ctx, B200H_E_INVALID, "etag requires B200H_MD5");
    const int device = b200h::ctx_device(ctx);
    std::vector<int> file_dev;
    std::string err;
    if (b200h::segment_devices(d_segs, seg_sizes, seg_of, n_files, file_dev, &err))
        return b200h::ctx_fail(ctx, B200H_E_INVALID, err);
    for (uint64_t i = 0; i < n_files; ++i)
        if (file_dev[i] >= 0 && file_dev[i] != device)
            return b200h::ctx_fail(ctx, B200H_E_INVALID, "file " + std::to_string(i) + " is on cuda:" +
                                                             std::to_string(file_dev[i]) + ", not on the context's cuda:" +
                                                             std::to_string(device));
    b200h::SegmentRows sr;
    b200h::segment_rows(d_segs, seg_sizes, seg_of, n_files, part_len, sr);
    const b200h::GatherRows gr{sr.piece_of.data(), sr.psrc.data(), sr.plen.data(), b200h::gather_cap()};
    return b200h::hash_device_rows(ctx, sr.addr.data(), sr.len.data(), sr.addr.size(), flags, sha256_out, md5_out,
                                   trimmed_len_out, sr.row_of.data(), n_files, etag_md5_out, &gr);
}

int b200h_segments_preview(const uint64_t* seg_sizes, const uint64_t* seg_of, uint64_t n_files, uint64_t part_len,
                           uint64_t window_bytes, uint64_t* n_rows_out, uint64_t* n_windows_out, uint8_t* gathered_out,
                           uint64_t* a_out, uint64_t* b_out, uint64_t* window_bytes_out) {
    if (n_files && !seg_of) return B200H_E_INVALID;
    for (uint64_t i = 0; i < n_files; ++i)
        if (seg_of[i] > seg_of[i + 1]) return B200H_E_INVALID;
    if (n_files && seg_of[n_files] > seg_of[0] && !seg_sizes) return B200H_E_INVALID;
    b200h::SegmentRows sr;
    b200h::segment_rows(nullptr, seg_sizes, seg_of, n_files, part_len, sr);
    const uint64_t rows = sr.len.size();
    std::vector<uint64_t> win, dst, wbytes;
    b200h::gather_windows(sr.len.data(), sr.piece_of.data(), rows, window_bytes ? window_bytes : b200h::gather_cap(),
                          win, dst, wbytes);
    if (n_rows_out) *n_rows_out = rows;
    if (n_windows_out) *n_windows_out = wbytes.size();
    if (window_bytes_out) std::copy(wbytes.begin(), wbytes.end(), window_bytes_out);
    for (uint64_t w = 0; w + 1 < win.size(); ++w)
        for (uint64_t r = win[w]; r < win[w + 1]; ++r) {
            const uint64_t pieces = sr.piece_of[r + 1] - sr.piece_of[r];
            if (gathered_out) gathered_out[r] = pieces != 0;
            if (a_out) a_out[r] = pieces ? w : sr.seg[r];
            if (b_out) b_out[r] = pieces ? pieces : sr.seg_off[r];
        }
    return 0;
}

}  // extern "C"
