// decode_kernels.cuh — launch interface of the decoder kernels (decode_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include "zb_decode.cuh"
#include "zb_blocks.cuh"

namespace zb {

#define EXEC_THREADS 128

// All pointers are device pointers.  dst_off must be non-decreasing with dst_off[i] + dst_cap[i] <= dst_off[i+1]
// (the scratch arenas are addressed from dst_off, see DESIGN.md "HBM layout").
struct DecodeArgs {
  const u8* src_base; const u64* src_off; const u32* src_size;
  u8* dst_base; const u64* dst_off; const u32* dst_cap;
  u32* result; u32 n;
  u32 item_base;       // index of item 0 within the arena numbering (slices of one batch share the arenas)
  FrameInfo* info;     // n records
  u8* lit_arena;       // decode_lit_arena_bytes()
  SeqRec* seq_arena;   // decode_seq_arena_bytes()
  // Items that hold several data frames (ZStdDecompress.cs:2096-2160) are decoded one data frame per pass: the
  // execute stage counts in *more the items that found another data frame behind the one it finished; the host
  // re-launches the pipeline with pass + 1 until the count stays 0.  Later passes skip every other item.
  const DictState* dict;   // the context's dictionary prepared by decode_load_dictionary (null: none), and its bytes
  const u8* dict_bytes;
  u32 pass;            // 0 = first data frame of every item
  u32* more;           // device counter, zeroed by the host before each pass (may be null: multi-frame items end after frame 1)
  // Block-parallel path for multi-block frames (zb_blocks.cuh).  units == nullptr switches it off.
  BlockUnit* units;    // decode_unit_arena_count() units; a slice uses the range that follows from its first dst_off / item_base
  u32* par_list;       // four lists of list_stride entries each (arena numbering, dense from [item_base]): the launch's FI_PAR items,
                       // then the items of the three sequence-kernel classes (FI_SEQ_A, FI_SEQ_B, full size)
  u32 list_stride;
  u32* cnt;            // eight device counters of this launch (zeroed by decode_launch): [0] units, [1] FI_PAR items, [2] FI_SMALLHUF,
                       // [3] FI_SEQ_A, [4] FI_SEQ_B, [5] full-size items of the frame-serial path (each the length of its list)
  u32 seq_a_max, seq_b_max;   // most sequences in a frame's first block for the sequence-kernel classes FI_SEQ_A / FI_SEQ_B (512 / 2 048;
                       // ZSTDB200_SEQ_A_MAX / _B_MAX let tests force wrong guesses and so the hand-over to the full-size kernel)
  u16* huf_full;       // decode_huf_full_bytes(decode_huf_ctas()) of scratch for the Huffman kernels of THIS launch (launches
                       // that run concurrently on different streams need regions of their own)
};

size_t decode_lit_arena_bytes(u64 max_dst_bytes, u64 max_items);
size_t decode_seq_arena_bytes(u64 max_dst_bytes, u64 max_items);
size_t decode_unit_arena_count(u64 max_dst_bytes, u64 max_items);
int decode_huf_ctas();                      // CTAs of one wave of k_huf / k_huf_blk (valid after decode_configure)
size_t decode_huf_full_bytes(int ctas);
cudaError_t decode_configure();
// parses the dictionary at d_dict_bytes (device memory, size bytes) into *d_state on `st` (one small kernel)
cudaError_t decode_load_dictionary(const u8* d_dict_bytes, u32 size, DictState* d_state, cudaStream_t st);
// enqueues the whole decode pipeline for one batch on `st`; *launches += number of kernels launched
cudaError_t decode_launch(const DecodeArgs& a, cudaStream_t st, int* launches, cudaEvent_t* marks = nullptr);
// marks (optional): DECODE_KERNELS + 1 events recorded before the first kernel and after each kernel
// (the block-parallel kernels k_huf_blk / k_seq_blk / k_exec_big run right after k_huf / k_seq / k_exec and are timed with them)
#define DECODE_KERNELS 5
extern const char* const kDecodeKernelNames[DECODE_KERNELS];

}  // namespace zb
