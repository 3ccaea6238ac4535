// b200hash_internal.h -- what a device group (b200hash_group.cu) needs from its member contexts beyond the C ABI.
#pragma once
#include <stddef.h>
#include <stdint.h>

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

}  // namespace b200h
