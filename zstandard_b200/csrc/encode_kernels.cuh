// encode_kernels.cuh — launch interface of the encoder kernels (encode_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <vector>
#include "host_plan.h"
#include "zb_common.cuh"

namespace zb {

struct EncDict;
struct DictState;

// All pointers are device pointers.  Item i: src_base[src_off[i] .. +src_size[i]) -> one zstd frame written at
// dst_base[dst_off[i] ..] (at most dst_cap[i] bytes); result[i] = frame size or an error code.
// src_off must be non-decreasing with src_off[i] + src_size[i] <= src_off[i+1] (the match stage's scratch is
// addressed from it) and the source buffer must be readable up to 8 bytes past its last item.
#define ENC_STREAM_PARTS 8
#define ENC_EXCLUSIVE 0xFFFFFFFFu

struct EncodeArgs {
  const u8* src_base; const u64* src_off; const u32* src_size;
  u8* dst_base; const u64* dst_off; const u32* dst_cap;
  u32* result; u32 n;
  u32 item_base;     // index of item 0 within the scratch numbering (slices of one batch share the arenas)
  int level, checksum;
  u32 max_src_size;  // largest src_size of the whole call (selects the match stage's table sizes, zb_encode.cuh enc_hlog_*)
  u32 stream_slot;   // partition (0..ENC_STREAM_PARTS-1) of the entropy stage's slot pool for launches that run concurrently
                     // on different streams, or ENC_EXCLUSIVE when the launch has the context to itself
  const EncDict* dict;   // the context's dictionary prepared for the encoder (zb_encode.cuh enc_dict_prepare), null: none
  u32 dict_id, dict_err; // its dictID and err, copied by the host (the entropy stage reads them from the parameter bank: no
                         // registers held across its frame loop)
};

// Per-device scratch owned by the context (allocated on the first compress call).
struct EncodeScratch {
  u8* lit = nullptr;       // literals of every block, addressed from src_off
  u32* seq = nullptr;      // sequence stores (2 words per sequence)
  void* meta = nullptr;    // per block: sequence and literal counts
  u8* slots = nullptr;     // entropy-stage work areas (code arrays, FSE state tables), one per resident thread
  u8* gtab = nullptr;      // match-stage hash tables of launches that have the device to themselves (allocated when first used)
  size_t maxBytes = 0, maxItems = 0;
  int sms = 148;
  u32 entWarps = 0;       // entropy-stage warps resident on the device at once (set with the arenas)
};

// The arguments of one launch over n items, numbered from item_base in the scratch, on stream slot `slot` (or ENC_EXCLUSIVE).
// dict: a block of enc_dict_block on the device, h_dict its host copy (for the id and error the launch carries); null: none.
EncodeArgs encode_args(const Items& it, size_t n, u32 item_base, int level, int checksum, u32 max_src_size, u32 slot,
                       const void* dict = nullptr, const std::vector<uint4>* h_dict = nullptr);
// dict_load on the host: what k_dict computes on the device (zb_format.cuh)
void dict_load_host(const u8* dict, u32 size, DictState& ds);
// The encoder's block of a dictionary (zb_encode.cuh EncDict, enc_dict_prepare) from its bytes and their DictState
std::vector<uint4> enc_dict_block(const u8* dict, u32 size, const DictState& ds);

size_t encode_bound(size_t srcSize);
cudaError_t encode_alloc(EncodeScratch& s, size_t maxBatchBytes, size_t maxItems);   // records sizes; memory comes lazily
void encode_free(EncodeScratch& s);
// marks (optional): ENCODE_KERNELS + 1 events recorded before the first kernel and after each kernel
#define ENCODE_KERNELS 3
extern const char* const kEncodeKernelNames[ENCODE_KERNELS];
cudaError_t encode_launch(const EncodeArgs& a, EncodeScratch& s, cudaStream_t st, int* launches, cudaEvent_t* marks = nullptr);
// Dictionary training: the match stage alone over items of at most one block (a.max_src_size <= 128 KiB) against a.dict, then
// the histograms of its literals and sequence codes added to stats[0..DT_STAT_WORDS) (zb_dict_train.cuh DtStats)
#define DT_STAT_WORDS (256 + 36 + 53 + 32)
cudaError_t encode_match_stats(const EncodeArgs& a, EncodeScratch& s, cudaStream_t st, u32* stats, int* launches);

}  // namespace zb
