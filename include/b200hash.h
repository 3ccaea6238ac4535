/*
 * b200hash.h -- C ABI of libb200hash.so: batched SHA-256 + MD5 content hashing on NVIDIA B200 (sm_100a).
 *
 * The reference (modal-labs/modal-client) has no FFI for this path: its seam is a set of Python
 * module-level functions that call hashlib.  Each entry point below names the reference call site(s)
 * it replaces (paths relative to the reference root).  INTEGRATION.md shows the ctypes stub a
 * maintainer would add to py/modal/_utils/hash_utils.py / blob_utils.py, and the cgo stub for go/blob.go.
 *
 * Conventions
 *   - every function returning int returns 0 on success and a negative B200H_E_* code on failure;
 *     b200h_last_error(ctx) gives a message (owned by the library, valid until the next call on ctx);
 *   - no exceptions cross the boundary; the caller owns every buffer it passes;
 *   - a context is bound to one CUDA device; batch calls on one context are serialised internally
 *     (thread-safe, re-entrant across contexts); the caller's GIL is never needed.  Concurrent SMALL
 *     b200h_hash_batch_host calls (<= 1024 messages each) are merged into one GPU batch by a combining queue
 *     (the first caller in leads, the others ride along and get their own rows back), and every b200h_stream
 *     runs on its own CUDA stream, so the reference's thread-pool callers overlap on the GPU;
 *   - there is NO CPU fallback: without a usable CUDA device b200h_create fails with B200H_E_CUDA.
 *   - digests are raw bytes: SHA-256 = 32 bytes (big-endian words, FIPS 180-4), MD5 = 16 bytes (RFC 1321).
 */
#ifndef B200HASH_H
#define B200HASH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200H_SHA256 1u     /* compute SHA-256 */
#define B200H_MD5 2u        /* compute MD5 */
#define B200H_TRIM_ZEROS 4u /* hash the prefix up to the last non-zero byte (volumefs2 blocks) */
#define B200H_HEX_OUT 32u /* the digest outputs receive lowercase ASCII hex (64 chars per SHA-256 row, 32 per MD5
                             row; buffers twice as wide) formatted on the device: the column MountFile.sha256_hex /
                             FileUploadSpec.md5_hex carry (modal_proto/api.proto:2582-2587), straight from the table */
#define B200H_NO_OUTLIERS 16u /* keep every message on the lane kernel (no outlier routing): with it
                                 b200h_hash_batch_device never reads anything back, i.e. only enqueues */

#define B200H_OK 0
#define B200H_E_INVALID (-1) /* bad argument */
#define B200H_E_CUDA (-2)    /* CUDA runtime / driver error (no device, launch failure, ...) */
#define B200H_E_NOMEM (-3)   /* host or device allocation failed */
#define B200H_E_STATE (-4)   /* object used in the wrong state (e.g. update after final) */
#define B200H_E_IO (-5)      /* a file could not be opened / read (b200h_stat_files, b200h_hash_files) */

typedef struct b200h_ctx b200h_ctx;
typedef struct b200h_stream b200h_stream;

/* ---- lifecycle ------------------------------------------------------------------------------- */

/* Bind a context to CUDA device `device`.  pinned_bytes / device_bytes size the host staging ring and
 * the HBM staging buffers used by the *_host entry points (0 = defaults: 512 MiB pinned, 8 GiB HBM,
 * both split in two for double buffering).  A message larger than one HBM wave slot is hashed in
 * consecutive segments with the chaining state kept on the device, so message size is not limited by them. */
int b200h_create(int device, size_t pinned_bytes, size_t device_bytes, b200h_ctx** out);
void b200h_destroy(b200h_ctx* ctx);
/* ctx may be NULL: returns the message of the last failed b200h_create on this thread. */
const char* b200h_last_error(b200h_ctx* ctx);
const char* b200h_version(void);
int b200h_device_count(void);

/* Page-locked host memory the *_host entry points can DMA from directly (no staging copy). */
void* b200h_host_alloc(b200h_ctx* ctx, size_t bytes);
void b200h_host_free(b200h_ctx* ctx, void* p);
/* The staging copy the *_host entry points use to fill their pinned ring: memcpy with non-temporal stores, widest
 * store the CPU has (AVX-512 / AVX2 / plain; picked once at run time, B200H_COPY_ISA caps the choice).  Exported for
 * callers that fill page-locked memory from b200h_host_alloc themselves (a serializer writing its output where the
 * DMA engine can take it) and for the CPU tests.  Needs no context and no GPU.  The reference has no counterpart. */
void b200h_stream_copy(void* dst, const void* src, size_t n);
const char* b200h_stream_copy_isa(void); /* "avx512" | "avx2" | "plain": what b200h_stream_copy runs on this CPU */

/* ---- batch hashing ---------------------------------------------------------------------------- */

/* Hash n independent messages that live in HOST memory; message i is base[offsets[i] .. +lengths[i]).
 * (base may be NULL with absolute addresses in offsets[].)  Outputs (each may be NULL): sha256_out[n*32],
 * md5_out[n*16], trimmed_len_out[n] (length actually hashed; == lengths[i] unless B200H_TRIM_ZEROS).
 * Stages through pinned memory to HBM with cudaMemcpyAsync in double-buffered waves; blocks until the
 * digests are in the output arrays.  The output arrays may be host or device memory (copied with
 * cudaMemcpyDefault): a caller that all-gathers the table over NCCL next passes device buffers.
 * Replaces: hashlib in hash_utils.get_upload_hashes (py/modal/_utils/hash_utils.py:68-101) as called per
 * payload from blob_utils.py:345 (map pump) and per file from blob_utils.py:459-474 (FileUploadSpec);
 * with B200H_TRIM_ZEROS: _find_end_of_block + _hash_range_sha256 (blob_utils.py:640-705);
 * md5.Sum/sha256.Sum256 in go/blob.go:51-52. */
int b200h_hash_batch_host(b200h_ctx* ctx, const uint8_t* base, const uint64_t* offsets, const uint64_t* lengths,
                          uint64_t n, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                          uint64_t* trimmed_len_out);

/* Same, but every pointer is a DEVICE pointer on ctx's device and the call only enqueues work on
 * `cuda_stream` (a cudaStream_t; NULL = the context's compute stream).  d_sha256/d_md5 must be 16-byte
 * aligned.  This is the HBM-resident path the roofline is quoted on.
 * Outlier routing (a few very long messages go to the chain kernel, whose launch is sized on the host) needs the
 * planner's count.  Three ways, in order of preference:
 *   b200h_hash_batch_device_hl  the caller also holds the lengths on the host (h_lengths[n] == d_lengths[n]): the
 *                               library computes the same selection there; the call ONLY ENQUEUES;
 *   flags | B200H_NO_OUTLIERS   no outlier routing for this batch (right for many similar messages); ONLY ENQUEUES;
 *   neither                     the count is read back after the ~12 us planning kernels: one synchronisation of
 *                               `cuda_stream` per call (also whenever B200H_TRIM_ZEROS is set and outliers are on:
 *                               the lengths that matter then exist on the device only). */
int b200h_hash_batch_device(b200h_ctx* ctx, const void* d_base, const uint64_t* d_offsets, const uint64_t* d_lengths,
                            uint64_t n, uint32_t flags, void* d_sha256, void* d_md5, uint64_t* d_trimmed_len,
                            void* cuda_stream);
int b200h_hash_batch_device_hl(b200h_ctx* ctx, const void* d_base, const uint64_t* d_offsets, const uint64_t* d_lengths,
                               const uint64_t* h_lengths, uint64_t n, uint32_t flags, void* d_sha256, void* d_md5,
                               uint64_t* d_trimmed_len, void* cuda_stream);

/* Split one host buffer into ceil(len/part_len) fixed-size parts and hash each (the last may be short).
 * etag_md5_out (may be NULL) = MD5 over the concatenated raw part MD5s, computed on the device
 * (requires B200H_MD5).  Returns the number of parts through *nparts_out.
 * Replaces: the per-8MiB-block loop of _gather_blocks (blob_utils.py:622-645, with B200H_TRIM_ZEROS) and
 * the per-part MD5 + md5(concat) ETag of perform_multipart_upload (blob_utils.py:194-219,
 * bytes_io_segment_payload.py:58,102). */
int b200h_hash_fixed_parts(b200h_ctx* ctx, const uint8_t* base, uint64_t len, uint64_t part_len, uint32_t flags,
                           uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out,
                           uint8_t etag_md5_out[16], uint64_t* nparts_out);

/* ---- buffers already in HBM, split into parts ------------------------------------------------------ */

/* The device-memory twin of b200h_hash_files(part_len): n buffers [d_bufs[i], +sizes[i]), each DEVICE memory on ctx's
 * device (any alignment), are hashed where they are.
 *   part_len == 0: one row per buffer (a zero-size buffer gives the empty-message digest);
 *   part_len  > 0: ceil(size/part_len) rows per buffer, flattened buffer-major (a zero-size buffer gives no rows);
 *                  with B200H_TRIM_ZEROS these are the volumefs2 blocks of a tensor's raw bytes.
 * Flags as for the host entry points (B200H_SHA256, B200H_MD5, B200H_TRIM_ZEROS, B200H_HEX_OUT).  etag_md5_out (n*16,
 * may be NULL; requires B200H_MD5): row i = MD5 over the concatenated raw part MD5s of buffer i, the multipart ETag of
 * b200h_hash_fixed_parts, computed on the device for every buffer in one more launch.  Outputs may be host or device
 * memory (cudaMemcpyDefault); the call returns when they are written.  The part table is built on the host and copied
 * once; nothing is read back except the planner's count when B200H_TRIM_ZEROS is set (see b200h_hash_batch_device).
 * A buffer that is not device memory on ctx's device is B200H_E_INVALID, last_error naming the buffer index and where
 * it lives.  Replaces: t.cpu() + a scratch file + the per-block reads of _gather_blocks / the whole-file hashlib
 * passes of _get_file_upload_spec for a tensor written to a Volume. */
int b200h_hash_device_parts(b200h_ctx* ctx, const void* const* d_bufs, const uint64_t* sizes, uint64_t n,
                            uint64_t part_len, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                            uint64_t* trimmed_len_out, uint8_t* etag_md5_out);

/* File i = the concatenation of segments [seg_of[i], seg_of[i+1]) (seg_of has n_files+1 entries, non-decreasing); every
 * non-empty segment is device memory on ctx's device, any alignment, any length (0 allowed).  Rows, flags and outputs
 * exactly as b200h_hash_device_parts over the concatenated bytes of each file: the rows are bit for bit those of
 * b200h_hash_device_parts on one buffer per file.  A safetensors file is one such file: its header, then its tensors.
 * A part that lies in one segment is hashed where it is.  A part that straddles segments (zero-size segments are not
 * boundaries) is gathered into a scratch buffer on ctx's device first, by one gather_pieces_kernel launch, and every
 * part of the call goes to the hash kernels in ONE batch -- a batch of 8 MiB blocks costs about one block's chain,
 * whatever the count.  Scratch holds every gathered part at once: at most min(file bytes, boundaries x part_len), and
 * with part_len == 0 a file of several non-empty segments is gathered whole.  The scratch is capped by
 * B200H_GATHER_BYTES (bytes, default 4 GiB): past the cap the gathered parts are hashed in successive windows (each
 * one gather + one batch), correct but slower; a single part larger than the cap is a window of its own.  The scratch
 * is allocated per call and freed before it returns; failing to allocate it is B200H_E_NOMEM, last_error giving the
 * size.  A segment that is not device memory on ctx's device is B200H_E_INVALID, last_error naming the file, the
 * segment index and where it lives. */
int b200h_hash_device_segments(b200h_ctx* ctx, const void* const* d_segs, const uint64_t* seg_sizes,
                               const uint64_t* seg_of, uint64_t n_files, uint64_t part_len, uint32_t flags,
                               uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out,
                               uint8_t* etag_md5_out);
/* The row table of b200h_hash_device_segments alone, from the sizes: no context, no GPU.  window_bytes 0 = the
 * B200H_GATHER_BYTES cap.  *n_rows_out = rows, *n_windows_out = windows (>= 1: contiguous row ranges, every window but
 * the first starting at a gathered row).  Per row r (arrays of n_rows, each may be NULL): gathered_out[r] = 0 for a
 * row hashed in place, with a_out[r] = its segment index and b_out[r] = its offset in that segment (an empty file's
 * one row: segment seg_of[i], offset 0); gathered_out[r] = 1 for a gathered row, with a_out[r] = its window and
 * b_out[r] = its number of pieces.  window_bytes_out[w] (n_windows entries, may be NULL) = scratch bytes of window w:
 * its gathered rows, each rounded up to 16 bytes.  Call with NULL arrays first to learn the counts.  Diagnostic. */
int b200h_segments_preview(const uint64_t* seg_sizes, const uint64_t* seg_of, uint64_t n_files, uint64_t part_len,
                           uint64_t window_bytes, uint64_t* n_rows_out, uint64_t* n_windows_out, uint8_t* gathered_out,
                           uint64_t* a_out, uint64_t* b_out, uint64_t* window_bytes_out);

/* ---- files (native reader pool; no Python I/O, no mmap) ------------------------------------------ */

/* Sizes (and permission bits, may be NULL) of n regular files, stat'ed by the library's I/O threads.
 * Replaces the per-file seek-to-end / os.stat of _get_file_upload_spec (blob_utils.py:455-457,494). */
int b200h_stat_files(b200h_ctx* ctx, const char* const* paths, uint64_t n, uint64_t* sizes_out, uint32_t* modes_out);

/* Hash the contents of n files.  The library's reader threads pread() them straight into the pinned staging
 * ring; waves are hashed while the next ones are being read.  sizes[] = what b200h_stat_files returned (a file
 * that turns out shorter is B200H_E_IO).
 *   part_len == 0: one message per file -> n rows (get_file_upload_spec_from_path over a tree:
 *                  py/modal/volume.py:1209-1216, py/modal/mount.py:467-485, blob_utils.py:490-501)
 *   part_len  > 0: every file is split into ceil(size/part_len) parts, rows flattened file-major; with
 *                  B200H_TRIM_ZEROS these are the volumefs2 blocks (blob_utils.py:622-645). */
int b200h_hash_files(b200h_ctx* ctx, const char* const* paths, uint64_t n, const uint64_t* sizes, uint64_t part_len,
                     uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out);

/* ---- streaming single message (hashlib-object shaped) ------------------------------------------- */

/* Incremental digest of ONE message fed in arbitrary pieces with bounded memory; the chaining state
 * stays on the device between updates.  A single message is a serial Merkle-Damgard chain, so this is
 * latency-bound by construction (~70 MB/s per stream) -- use the batch entry points for throughput.
 * update() gathers into a pinned buffer and enqueues one absorb per 4 MiB (B200H_STREAM_BUF) without waiting
 * for it; every stream has its own CUDA stream and scratch, so N streams fed from N threads advance concurrently.
 * One stream object must not be used from two threads at once (like a hashlib object).
 * Replaces: hashlib objects in hash_utils._update over a BinaryIO (hash_utils.py:18-29) and
 * BytesIOSegmentPayload._md5_checksum (bytes_io_segment_payload.py:58,102,79-80). */
int b200h_stream_new(b200h_ctx* ctx, uint32_t flags, b200h_stream** out);
int b200h_stream_update(b200h_stream* s, const uint8_t* data, uint64_t len);
/* Non-destructive: may be called repeatedly and interleaved with further updates (like hashlib.digest()). */
int b200h_stream_digest(b200h_stream* s, uint8_t sha256_out[32], uint8_t md5_out[16]);
int b200h_stream_reset(b200h_stream* s);
void b200h_stream_free(b200h_stream* s);

/* ---- dedupe of the digest table (the step right after the path) ---------------------------------- */

/* For n fixed-width keys (key_bytes = 32: SHA-256 rows, 16: MD5 rows) compute first[i] = the smallest j with
 * key_j == key_i (so first[i] == i marks the first occurrence of a content) and the number of distinct keys.
 * Exact (full-key comparison), deterministic, computed on the device over a hash table in HBM.
 * Replaces: the `accounted_hashes` set of _Mount._load_mount (py/modal/mount.py:498,518-534), which dedupes one
 * file at a time on the event loop, and the per-file MountPutFile existence round trips the volumefs1 uploader
 * spends on duplicates inside one batch (py/modal/volume.py:1288-1296).
 * _host: keys / first_out are host arrays, blocks until done.  _device: every pointer is a device pointer
 * (d_keys 4-byte aligned, d_ndistinct may be NULL), work is only enqueued on cuda_stream (NULL = ctx's stream). */
int b200h_dedupe_host(b200h_ctx* ctx, const uint8_t* keys, uint64_t n, uint32_t key_bytes, uint32_t* first_out,
                      uint64_t* ndistinct_out);
int b200h_dedupe_device(b200h_ctx* ctx, const void* d_keys, uint64_t n, uint32_t key_bytes, uint32_t* d_first,
                        uint64_t* d_ndistinct, void* cuda_stream);

/* ---- utilities ---------------------------------------------------------------------------------- */

/* Counter-based synthetic bytes on the device (bench / test data): d_dst[0..nbytes) = bytes
 * [start, start+nbytes) of stream `seed`; d_dst 8-byte aligned, start a multiple of 8. */
int b200h_fill_synth_device(b200h_ctx* ctx, void* d_dst, uint64_t nbytes, uint64_t seed, uint64_t start,
                            void* cuda_stream);
/* How many messages of the most recent batch the planner handed to the outlier path (chain kernel: one CTA per
 * long message) instead of the lane kernel.  Diagnostic. */
int b200h_last_outlier_count(b200h_ctx* ctx, uint32_t* count_out);
/* The staging step of b200h_hash_batch_host on its own: gather n messages (base may be NULL with absolute addresses in
 * offsets[]) into dst the way a wave is laid out in HBM -- message i at the next multiple of 16, offsets returned
 * through packed_offsets_out -- with the library's packer team of `threads` threads working slot_bytes at a time (the
 * size of a pinned slot).  dst needs sum((len + 15) & ~15) bytes.  No context, no GPU: for the CPU tests of the packer
 * and for measuring a host's packing rate (tools/packbench.py).  Diagnostic. */
int b200h_pack_preview(const uint8_t* base, const uint64_t* offsets, const uint64_t* lengths, uint64_t n, uint8_t* dst,
                       uint64_t dst_bytes, uint64_t slot_bytes, int threads, uint64_t* packed_offsets_out);
/* What the planner decides for a batch with these message lengths on a device with sm_count SMs (default settings):
 * how many messages go to the chain kernel (true outliers, DESIGN.md 5.4) and how many form the long lane queue
 * (second, lane-packed launch, DESIGN.md 5.3).  Pure host arithmetic -- the same code that sizes the launches of
 * b200h_hash_batch_host / _device_hl without reading the device planner's answer back -- so it needs neither a
 * context nor a GPU.  flags: B200H_SHA256 / B200H_MD5 / B200H_NO_OUTLIERS.  Diagnostic. */
int b200h_plan_preview(const uint64_t* lengths, uint64_t n, uint32_t flags, uint32_t sm_count, uint32_t* n_chain_out,
                       uint32_t* n_long_out);
/* Kernels launched by this context so far (all kinds). */
uint64_t b200h_launch_count(b200h_ctx* ctx);
/* Combining queue of b200h_hash_batch_host: GPU batches issued for, and caller requests served by, the small-request
 * path so far (requests / groups = how many concurrent callers shared a batch on average). */
int b200h_combine_stats(b200h_ctx* ctx, uint64_t* groups_out, uint64_t* requests_out);
/* Enqueues that had to synchronise their stream to read the planner's outlier count back (see
 * b200h_hash_batch_device); 0 for a caller that passes host lengths or B200H_NO_OUTLIERS. */
uint64_t b200h_plan_sync_count(b200h_ctx* ctx);
/* When enabled, every lane_hash launch is bracketed by CUDA events on its stream;
 * b200h_profile_read synchronises and returns the accumulated device time and launch count, then clears. */
int b200h_profile_enable(b200h_ctx* ctx, int on);
int b200h_profile_read(b200h_ctx* ctx, double* hash_kernel_ms, uint64_t* hash_kernel_launches);

/* ---- device groups: one process, several GPUs ------------------------------------------------------ */

/* A group is one context per listed device (a device may repeat: {0, 0} is two contexts on one GPU), driven as one.
 * b200h_group_hash_batch_host / _hash_files deal a batch over the members by bytes (b200h_group_split_preview), every
 * member hashes its share on its own thread at the same time, and the rows land at the caller's message indices.
 * Members on one NUMA node divide its CPUs between their packer and reader teams.  Group calls are thread-safe.
 * b200h_group_hash_device_parts deals the parts of buffers already in HBM over the members on each buffer's device.
 * Everything else (stat_files, dedupe_*, hash_fixed_parts, streams, host_alloc, the *_device entry points) is not
 * split: call it on b200h_group_member(g, 0), the "home" member.  Its host_alloc memory is portable, so every member
 * DMAs it directly. */
typedef struct b200h_group b200h_group;

/* min_share_bytes: a batch is split over k = min(members, messages, max(1, total bytes / min_share_bytes)) members
 * (0 = the default, B200H_GROUP_MIN_SHARE).  pinned_bytes / device_bytes size every member as in b200h_create. */
#define B200H_GROUP_MIN_SHARE (256ull << 20)
int b200h_group_create(const int* devices, int ndevices, size_t pinned_bytes, size_t device_bytes,
                       uint64_t min_share_bytes, b200h_group** out);
void b200h_group_destroy(b200h_group* g);
/* g may be NULL: the message of the last failed b200h_group_create on this thread.  A failed batch names the first
 * failing member ("member 1 (cuda:0): ..."); the other members finish their shares, the outputs are unspecified and
 * the group stays usable. */
const char* b200h_group_last_error(b200h_group* g);
int b200h_group_size(b200h_group* g);
b200h_ctx* b200h_group_member(b200h_group* g, int i); /* owned by the group; member 0 = "home" */
/* As b200h_hash_batch_host.  With k == 1 this IS that call on the home member (combining queue included).  Outputs
 * may be host or device memory; device outputs must all be on one device (the table device), B200H_E_INVALID
 * otherwise: each member hashes into its own HBM and scatter_rows_kernel writes its rows into the table, over peer
 * access where the devices allow it (enabled for this process's contexts only), else after a cudaMemcpyPeerAsync. */
int b200h_group_hash_batch_host(b200h_group* g, const uint8_t* base, const uint64_t* offsets, const uint64_t* lengths,
                                uint64_t n, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                                uint64_t* trimmed_len_out);
/* As b200h_hash_files; with part_len > 0 the parts are dealt, so one file's blocks may land on several members. */
int b200h_group_hash_files(b200h_group* g, const char* const* paths, uint64_t n, const uint64_t* sizes,
                           uint64_t part_len, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                           uint64_t* trimmed_len_out);
/* As b200h_hash_device_parts.  A buffer is only hashed by members on the device that holds it: the parts resident on
 * device d are dealt over the members on d by the rule above, so {0, 0} splits one GPU's parts and {0, 1} hashes each
 * GPU's buffers on that GPU.  Every member works on its own thread and the rows land at their global indices; ETags
 * are computed after all MD5 rows are in place.  A buffer on a device with no member is B200H_E_INVALID ("buffer 3 is
 * on cuda:5, which is not in the group"); the group stays usable.  When one member takes the whole batch this IS
 * b200h_hash_device_parts on that member. */
int b200h_group_hash_device_parts(b200h_group* g, const void* const* d_bufs, const uint64_t* sizes, uint64_t n,
                                  uint64_t part_len, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                                  uint64_t* trimmed_len_out, uint8_t* etag_md5_out);
/* As b200h_hash_device_segments.  Every file's non-empty segments must be on one device ("file 2 has segments on
 * cuda:0 and cuda:1" otherwise, B200H_E_INVALID; the group stays usable).  The rows of the files on device d are dealt
 * over the members on d as in b200h_group_hash_device_parts; a member gathers the straddling rows of its own share into
 * its own scratch (capped per member by B200H_GATHER_BYTES).  When one member takes the whole batch this IS
 * b200h_hash_device_segments on that member. */
int b200h_group_hash_device_segments(b200h_group* g, const void* const* d_segs, const uint64_t* seg_sizes,
                                     const uint64_t* seg_of, uint64_t n_files, uint64_t part_len, uint32_t flags,
                                     uint8_t* sha256_out, uint8_t* md5_out, uint64_t* trimmed_len_out,
                                     uint8_t* etag_md5_out);
/* What the last batch call did, per member (arrays of b200h_group_size entries, each may be NULL): messages, payload
 * bytes, bytes that went through the member's pinned staging ring (0 = DMAed straight from the caller's page-locked
 * memory) and wall milliseconds spent inside the member.  Members the batch did not use report zeros. */
int b200h_group_last_split(b200h_group* g, uint64_t* messages_out, uint64_t* bytes_out, uint64_t* staged_bytes_out,
                           double* busy_ms_out);
/* The split decision alone: owner_out[n] = member of every message, *members_used_out = k.  Messages are sorted by
 * length (longest first, stable) and dealt over members 0..k-1 in boustrophedon order (0..k-1, k-1..0, ...).  Pure
 * host arithmetic: no group, no GPU.  min_share_bytes 0 = B200H_GROUP_MIN_SHARE. */
int b200h_group_split_preview(const uint64_t* lengths, uint64_t n, int nmembers, uint64_t min_share_bytes,
                              uint32_t* owner_out, int* members_used_out);

#ifdef __cplusplus
}
#endif
#endif /* B200HASH_H */
