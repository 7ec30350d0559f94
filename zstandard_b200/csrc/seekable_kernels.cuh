// seekable_kernels.cuh — launch interface of the seekable-archive kernels (seekable_kernels.cu, format in seekable.h).
#pragma once
#include <cuda_runtime.h>
#include "host_plan.h"
#include "zb_common.cuh"

namespace zb {

// Pack: frame i (an encoder result) lies at frames[frame_off[i] ..], 16-byte aligned, result[i] bytes long, and holds
// content[i] bytes of input.  The frames are moved back to back to out[0 ..).  With table != 0 the seek table follows them
// (entries from the sizes and, with checksum != 0, each frame's own 4-byte trailer) and *dst_size gets the archive's size.
// offsets: n + 2 words of device scratch (the exclusive scan).  A frame with an error result packs nothing: *dst_size = 0.
struct SeekPackArgs {
  const u8* frames; const u64* frame_off; const u32* result; const u32* content; u32 n;
  u8* out; u64* offsets; u64* dst_size; int table, checksum;
};
cudaError_t seek_pack(const SeekPackArgs& a, cudaStream_t st, int* launches);

// Check: item i of `it` was decoded (FrameInfo info[i], with DecodeArgs::more null) against a table entry whose
// Decompressed_Size is it.dstCap[i] (the capacity it was given) and, when cksum != null, whose Checksum is cksum[i].
// result[i] becomes corruption_detected when the size differs (a capacity too small means it does) or when another data
// frame follows the first inside the entry's Compressed_Size; checksum_wrong when the checksum does not match (a frame's own
// checksum is read at info[i].trailer_off, where the decoder verified it).  With first != null the error of the lowest archive
// frame index (frame[i]) is kept in *first as (index << 32 | code); after the last block of `blocks_total`
// (over every check launch since *first = ~0 and *done = 0), *code = that code, or `preset` when no frame failed.
struct SeekCheckArgs {
  Items it; const FrameInfo* info; u32 n; const u32* cksum; const u32* frame;
  unsigned long long* first; u32* done; u32 blocks_total; u32* code; u32 preset;
};
constexpr u32 SEEK_CHECK_WARPS = 8;   // frames per block of k_seek_check
inline u32 seek_check_blocks(u32 n) { return n ? (n + SEEK_CHECK_WARPS - 1) / SEEK_CHECK_WARPS : 1; }
cudaError_t seek_check(const SeekCheckArgs& a, cudaStream_t st, int* launches);

}  // namespace zb
