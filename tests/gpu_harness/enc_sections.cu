// enc_sections.cu — test harness: the entropy stage's section writers (zb_encode_warp.cuh) on crafted blocks, one warp per case.
//
// Each case is a block's literals and sequence store (the u32-pair format of SeqStore, bits 30 / 31 of the second word included),
// a level and a capacity.  A warp writes the literals section with warp_enc_literals (no dictionary; raw only at the negative
// levels) and, when that fits, the sequences section with warp_enc_sequences on the rest of the room, as k_enc_entropy calls
// them.  The serial writers of tests/hostsim/serial_encoder.h are run on the same layout by tests/hostsim/enc_sections.cpp.
//
// Case descriptor, 8 u64 per case:
//   [0] literal offset into lits   [1] literal count   [2] sequence offset into seqs (u32 words, a multiple of 2)   [3] nbSeq
//   [4] level (two's complement)   [5] capacity        [6] offset of the case's region in out (a multiple of 16)   [7] misalign
// The section is written at out + [6] + 64 + [7]; the caller surrounds [out, out + capacity) with sentinel bytes and checks
// afterwards that none of them changed.  sizes[2 i], sizes[2 i + 1]: bytes of the literals / sequences section (0 = no room).
#include "../../zstandard_b200/csrc/zb_encode_warp.cuh"
#include <cuda_runtime.h>

namespace zb {

__global__ void __launch_bounds__(32) k_enc_sections(u32 n, const u64* desc, const u8* lits, const u32* seqs, u8* out, u32* sizes, u8* slots) {
  __shared__ EntWarp w;
  __shared__ EntLut lut;
  const u32 lane = threadIdx.x;
  lut.ll[lane] = ll_info(lane);
  if (lane < 36 - 32) lut.ll[32 + lane] = ll_info(32 + lane);
  lut.ml[lane] = ml_info(lane);
  if (lane < 53 - 32) lut.ml[32 + lane] = ml_info(32 + lane);
  __syncwarp();
  u8* const codes = slots + (size_t)blockIdx.x * slot_bytes();
  u8* const tmp = codes + align16((size_t)kBlockSeqCap * 3);
  for (u32 c = blockIdx.x; c < n; c += gridDim.x) {
    const u64* d = desc + 8 * (size_t)c;
    SeqStore st;
    st.lits = const_cast<u8*>(lits + d[0]); st.nlits = (u32)d[1];
    st.seqs = const_cast<u32*>(seqs + d[2]); st.n = (u32)d[3]; st.cap = kBlockSeqCap;
    const int level = (int)(i64)d[4];
    const u32 cap = (u32)d[5];
    u8* const body = out + d[6] + 64 + d[7];
    const u32 l = warp_enc_literals(body, cap, st.lits, st.nlits, w, tmp, lane, nullptr, level < 0);
    u32 s = 0;
    if (l) s = warp_enc_sequences(body + l, cap - l, st, codes, w, lut, level, lane, nullptr);
    if (lane == 0) { sizes[2 * c] = l; sizes[2 * c + 1] = s; }
    __syncwarp();
  }
}

}  // namespace zb

// Host entry: copies the cases in, runs them, copies out (in place) and sizes back.  Returns a cudaError_t.
extern "C" int enc_sections_run(unsigned n, const unsigned long long* desc, const unsigned char* lits, unsigned long long litBytes,
                                const unsigned* seqs, unsigned long long seqWords, unsigned char* out, unsigned long long outBytes,
                                unsigned* sizes) {
  using namespace zb;
  const u32 warps = n < 1024 ? n : 1024;
  u64* dDesc = nullptr; u8* dLits = nullptr; u32* dSeqs = nullptr; u8* dOut = nullptr; u32* dSizes = nullptr; u8* dSlots = nullptr;
  cudaError_t e = cudaSuccess;
  if (n == 0) return 0;
  if ((e = cudaMalloc(&dDesc, 64 * (size_t)n)) != cudaSuccess || (e = cudaMalloc(&dLits, litBytes + 64)) != cudaSuccess ||
      (e = cudaMalloc(&dSeqs, 4 * seqWords + 64)) != cudaSuccess || (e = cudaMalloc(&dOut, outBytes)) != cudaSuccess ||
      (e = cudaMalloc(&dSizes, 8 * (size_t)n)) != cudaSuccess || (e = cudaMalloc(&dSlots, (size_t)warps * slot_bytes())) != cudaSuccess)
    goto done;
  if ((e = cudaMemcpy(dDesc, desc, 64 * (size_t)n, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(dLits, lits, litBytes, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(dSeqs, seqs, 4 * seqWords, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(dOut, out, outBytes, cudaMemcpyHostToDevice)) != cudaSuccess)
    goto done;
  k_enc_sections<<<warps, 32>>>(n, dDesc, dLits, dSeqs, dOut, dSizes, dSlots);
  if ((e = cudaGetLastError()) != cudaSuccess || (e = cudaDeviceSynchronize()) != cudaSuccess) goto done;
  if ((e = cudaMemcpy(out, dOut, outBytes, cudaMemcpyDeviceToHost)) != cudaSuccess ||
      (e = cudaMemcpy(sizes, dSizes, 8 * (size_t)n, cudaMemcpyDeviceToHost)) != cudaSuccess)
    goto done;
done:
  cudaFree(dDesc); cudaFree(dLits); cudaFree(dSeqs); cudaFree(dOut); cudaFree(dSizes); cudaFree(dSlots);
  return (int)e;
}
