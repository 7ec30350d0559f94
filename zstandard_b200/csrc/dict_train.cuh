// dict_train.cuh — host interface of the dictionary trainer (dict_train.cu) for api.cu.
#pragma once
#include <cuda_runtime.h>
#include <string>
#include "../../include/zstdb200.h"
#include "encode_kernels.cuh"

namespace zb {

// What a training call borrows from the context's first device: its encoder arenas and the staging of the host-pointer path
// (the call is synchronous and a context is single-caller, so nothing else uses them meanwhile).
struct DtDevice {
  cudaStream_t stream;
  EncodeScratch* enc;
  u8* d_dst; size_t dstCap;          // compressed output of the scoring passes
  u32* d_result; u32* h_result;      // their result codes (maxItems)
  u8* d_desc; u8* h_desc;            // descriptors, maxItems x 24 bytes each side
  size_t maxBatch, maxItems;
  uint64_t launches;
};

// zstdb200_train_dictionary on the current device.  Returns the dictionary size or an error code (GENERIC: err says why).
u32 dt_train_run(DtDevice& dv, u8* dict, u32 capacity, const u8* samples, const u32* sizes, size_t n, zstdb200_train_params& pr,
                 std::string& err);

}  // namespace zb
