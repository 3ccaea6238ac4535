// b200hash_internal.h -- what a device group (b200hash_group.cu) and the device-buffer entry points
// (b200hash_device_parts.cu) need from a context beyond the C ABI.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../include/b200hash.h"

namespace b200h {

// b200h_create for one member of a device group.  group_devices[ngroup] are the devices of every member (repeats
// allowed); the members on this device's NUMA node divide its CPUs between their packer and reader teams, the way
// LOCAL_WORLD_SIZE ranks do.  ngroup <= 1 is exactly b200h_create.
int create_member(int device, size_t pinned_bytes, size_t device_bytes, const int* group_devices, int ngroup,
                  b200h_ctx** out);

// One member's share of a group batch: b200h_hash_batch_host without the combining queue (paths == NULL), or the
// messages of b200h_hash_files (paths[file_of[i]] at byte offset off[i]).  A share dealt from a batch in page-locked
// memory is sparse; its large messages are DMAed one by one instead of being re-staged.  *staged_out = bytes that
// went through the pinned staging ring.
int hash_share(b200h_ctx* ctx, const uint8_t* base, const uint64_t* off, const uint64_t* len, uint64_t n, uint32_t flags,
               uint8_t* sha_out, uint8_t* md5_out, uint64_t* trim_out, const char* const* paths, const uint64_t* file_of,
               uint64_t* staged_out);

// Bytes ctx has put through its pinned staging ring so far (all calls).
uint64_t staged_bytes(b200h_ctx* ctx);

// The message list of b200h_hash_files: one per file (part_len == 0) or one per part_len-sized part, file-major.
void file_messages(const uint64_t* sizes, uint64_t n, uint64_t part_len, std::vector<uint64_t>& off,
                   std::vector<uint64_t>& len, std::vector<uint64_t>& file_of);

// ---- device-resident buffers (b200hash_device_parts.cu) ----

// The CUDA device ctx is bound to, and ctx's last_error set to msg (returns code).
int ctx_device(b200h_ctx* ctx);
int ctx_fail(b200h_ctx* ctx, int code, const std::string& msg);

// Where [d_bufs[i], +sizes[i]) lives: the device index, or -1 with *what set ("host memory", ...) when it is not
// device memory.  A zero-size buffer is nowhere (returns -2) and may be any pointer.
int buffer_device(const void* p, uint64_t size, std::string* what);

// The row table of b200h_hash_device_parts: absolute device addresses and lengths of every part, file-major, and the
// first row of every buffer (row_of[n] = rows).
void device_part_rows(const void* const* d_bufs, const uint64_t* sizes, uint64_t n, uint64_t part_len,
                      std::vector<uint64_t>& addr, std::vector<uint64_t>& len, std::vector<uint64_t>& row_of);

// ---- files made of device segments (b200hash_device_segments.cu) ----

// Rows whose bytes straddle segments: row r is gathered when piece_of[r + 1] > piece_of[r], and then consists of the
// pieces (psrc[p], plen[p]) for p in [piece_of[r], piece_of[r + 1]), in order.  The gathered rows are copied into
// scratch in windows of at most window_bytes (16-byte aligned rows; a longer row is a window of its own).
struct GatherRows {
    const uint64_t* piece_of;
    const uint64_t* psrc;
    const uint64_t* plen;
    uint64_t window_bytes;
};

// The row table of b200h_hash_device_segments.  In-place rows: addr (absolute), seg / seg_off (segment index and
// offset in it); gathered rows: their pieces.  An empty file's one row (part_len 0) is in place at (seg_of[i], 0).
struct SegmentRows {
    std::vector<uint64_t> addr, len, seg, seg_off, piece_of, psrc, plen, row_of;
};
// d_segs may be NULL (addresses from 0: the host preview).
void segment_rows(const void* const* d_segs, const uint64_t* seg_sizes, const uint64_t* seg_of, uint64_t n_files,
                  uint64_t part_len, SegmentRows& out);
// Windows = contiguous row ranges [win[w], win[w + 1]); each window after the first starts at a gathered row.
// dst[r] = offset of gathered row r in its window's scratch, win_bytes[w] = scratch bytes window w needs.
void gather_windows(const uint64_t* len, const uint64_t* piece_of, uint64_t rows, uint64_t window_bytes,
                    std::vector<uint64_t>& win, std::vector<uint64_t>& dst, std::vector<uint64_t>& win_bytes);
// file_dev[i] = device of file i's non-empty segments (-2: it has none).  -1 with *err set when a segment is not
// device memory or a file's segments are on two devices.
int segment_devices(const void* const* d_segs, const uint64_t* seg_sizes, const uint64_t* seg_of, uint64_t n_files,
                    std::vector<int>& file_dev, std::string* err);
// "" or what is wrong with the pointer / seg_of arguments of a segments call.
std::string segment_args_error(const void* const* d_segs, const uint64_t* seg_sizes, const uint64_t* seg_of,
                               uint64_t n_files);
// B200H_GATHER_BYTES, default 4 GiB: the scratch cap per call (per member in a group).
uint64_t gather_cap();
// Pieces longer than this are split into several work items of gather_pieces_kernel.
uint64_t gather_item_bytes();
// gather_pieces_kernel over `items` work items (device arrays src | dst | len) on st; returns the launches made.
int launch_gather(const uint64_t* d_src, const uint64_t* d_dst, const uint64_t* d_len, uint64_t items, cudaStream_t st);

// Hash `rows` device-resident messages (absolute addresses, on ctx's device; a zero-length row may hold any address)
// on ctx: the row table goes to the device in one copy, then trim -> plan -> lane/chain on the context's stream with
// the lengths known on the host.  etag_out (n*16, may be NULL) = MD5 over the raw MD5 rows [row_of[i], row_of[i+1])
// of buffer i, one more lane_hash launch.  Outputs may be host or device memory; returns when they are written.
// gather (may be NULL): rows to copy into scratch first (their addr[] is ignored).  With one window every row is in
// one batch; with several, window w's gather and its rows' batch run in turn on the context's stream.
int hash_device_rows(b200h_ctx* ctx, const uint64_t* addr, const uint64_t* len, uint64_t rows, uint32_t flags,
                     uint8_t* sha_out, uint8_t* md5_out, uint64_t* trim_out, const uint64_t* row_of, uint64_t n,
                     uint8_t* etag_out, const GatherRows* gather = nullptr);

// rows x width raw digest bytes in host memory -> lowercase hex rows (2 x width) at out (host or device), formatted
// on ctx's device.
int hex_rows_from_host(b200h_ctx* ctx, const uint8_t* raw, uint64_t nbytes, uint8_t* out);

}  // namespace b200h
