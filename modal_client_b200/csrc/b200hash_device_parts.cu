// b200hash_device_parts.cu -- b200h_hash_device_parts: buffers that already live in HBM, split into parts and hashed
// where they are (C ABI: include/b200hash.h).  The device-memory twin of b200h_hash_files(part_len): the part table
// is built here on the host, where the lengths are, and the work runs on the context's plan -> trim -> lane/chain
// kernels (hash_device_rows in b200hash_api.cu).  The group form is b200h_group_hash_device_parts
// (b200hash_group.cu), which deals the parts of every device over the members on that device.
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/b200hash.h"
#include "b200hash_internal.h"

int b200h::buffer_device(const void* p, uint64_t size, std::string* what) {
    if (size == 0) return -2;
    const uint8_t* ends[2] = {(const uint8_t*)p, (const uint8_t*)p + (size - 1)};
    int dev = -1;
    for (int k = 0; k < 2; ++k) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, ends[k]) != cudaSuccess) {
            cudaGetLastError();
            *what = "not memory CUDA knows";
            return -1;
        }
        if (at.type != cudaMemoryTypeDevice) {
            *what = k ? "device memory that ends outside device memory"
                      : (at.type == cudaMemoryTypeManaged ? "managed memory"
                         : at.type == cudaMemoryTypeHost  ? "page-locked host memory"
                                                          : "host memory");
            return -1;
        }
        if (k && at.device != dev) {
            *what = "a range that spans two devices";
            return -1;
        }
        dev = at.device;
    }
    return dev;
}

void b200h::device_part_rows(const void* const* d_bufs, const uint64_t* sizes, uint64_t n, uint64_t part_len,
                             std::vector<uint64_t>& addr, std::vector<uint64_t>& len, std::vector<uint64_t>& row_of) {
    std::vector<uint64_t> off, file_of;
    b200h::file_messages(sizes, n, part_len, off, len, file_of);
    addr.resize(off.size());
    for (size_t r = 0; r < off.size(); ++r) addr[r] = (uint64_t)(uintptr_t)d_bufs[file_of[r]] + off[r];
    row_of.assign(n + 1, 0);
    for (size_t r = 0; r < file_of.size(); ++r) row_of[file_of[r] + 1] += 1;
    for (uint64_t b = 0; b < n; ++b) row_of[b + 1] += row_of[b];
}

extern "C" {

int b200h_hash_device_parts(b200h_ctx* ctx, const void* const* d_bufs, const uint64_t* sizes, uint64_t n,
                            uint64_t part_len, uint32_t flags, uint8_t* sha256_out, uint8_t* md5_out,
                            uint64_t* trimmed_len_out, uint8_t* etag_md5_out) {
    if (!ctx) return B200H_E_INVALID;
    if (n && (!d_bufs || !sizes)) return b200h::ctx_fail(ctx, B200H_E_INVALID, "d_bufs/sizes must not be NULL");
    if (!(flags & (B200H_SHA256 | B200H_MD5)))
        return b200h::ctx_fail(ctx, B200H_E_INVALID, "flags select neither SHA256 nor MD5");
    if (etag_md5_out && !(flags & B200H_MD5)) return b200h::ctx_fail(ctx, B200H_E_INVALID, "etag requires B200H_MD5");
    const int device = b200h::ctx_device(ctx);
    for (uint64_t i = 0; i < n; ++i) {
        std::string what;
        const int d = b200h::buffer_device(d_bufs[i], sizes[i], &what);
        if (d == -1) return b200h::ctx_fail(ctx, B200H_E_INVALID, "buffer " + std::to_string(i) + " is " + what);
        if (d >= 0 && d != device)
            return b200h::ctx_fail(ctx, B200H_E_INVALID, "buffer " + std::to_string(i) + " is on cuda:" + std::to_string(d) +
                                                             ", not on the context's cuda:" + std::to_string(device));
    }
    std::vector<uint64_t> addr, len, row_of;
    b200h::device_part_rows(d_bufs, sizes, n, part_len, addr, len, row_of);
    return b200h::hash_device_rows(ctx, addr.data(), len.data(), addr.size(), flags, sha256_out, md5_out,
                                   trimmed_len_out, row_of.data(), n, etag_md5_out);
}

}  // extern "C"
