/* zmt_dev.h — internal alias of the public device-level header, plus what only the library itself calls. */
#pragma once
#include "../../include/zstdmt_b200_dev.h"

/* zmt_zstd_scan_frame_host for a frame whose length is not known in advance (plain .zst streams): *consumed receives
 * the frame length and bytes after the frame are not an error. */
extern "C" int zmt_zstd_scan_frame_host2(const uint8_t* frame, size_t n, uint64_t base_off, uint32_t frame_idx, void* blocks_out, uint32_t* nblocks_io,
                                         uint32_t max_blocks, uint64_t* scratch_used, uint64_t* content_size, uint32_t* needs_seq, size_t* consumed);
