// exec_copy.cu — test harness: the execute stage's flattened copies (zb_exec_copy.cuh) on described sets of runs, one warp
// per case, called as k_exec and k_exec_big call them for one group of 32 sequences.
//
// Case descriptor, 4 u64 per case:
//   [0] kind: 0 literal copy (flat_literals), 1 RLE fill (flat_literals with isRle), 2 match copy (flat_matches)
//   [1] offset of the group's first byte g in buf     [2] offset of the literal base in lits     [3] the RLE byte
// Runs, 3 u32 per lane (32 lanes per case): destination position relative to g, then the source position relative to
// the literal base (kind 0) or the match offset (kind 2, the source is g + dpos - off), then the length (0: no run).
#include "../../zstandard_b200/csrc/zb_exec_copy.cuh"
#include <cuda_runtime.h>

namespace zb {

__global__ void __launch_bounds__(32) k_exec_copy(u32 n, const u64* desc, const u32* runs, const u8* lits, u8* buf) {
  const u32 lane = threadIdx.x;
  for (u32 c = blockIdx.x; c < n; c += gridDim.x) {
    const u64* d = desc + 4 * (size_t)c;
    const u32* r = runs + 96 * (size_t)c + 3 * lane;
    u8* const g = buf + d[1];
    if (d[0] == 2) flat_matches(g, r[0], r[1], r[2], lane);
    else flat_literals(g, lits + d[2], d[0] == 1, (u32)d[3], r[0], r[1], r[2], lane);
    __syncwarp();
  }
}

}  // namespace zb

// Host entry: copies the cases and buf in, runs them, copies buf back in place.  Returns a cudaError_t.
extern "C" int exec_copy_run(unsigned n, const unsigned long long* desc, const unsigned* runs, const unsigned char* lits,
                             unsigned long long litBytes, unsigned char* buf, unsigned long long bufBytes) {
  using namespace zb;
  u64* dDesc = nullptr; u32* dRuns = nullptr; u8* dLits = nullptr; u8* dBuf = nullptr;
  cudaError_t e = cudaSuccess;
  if (n == 0) return 0;
  if ((e = cudaMalloc(&dDesc, 32 * (size_t)n)) != cudaSuccess || (e = cudaMalloc(&dRuns, 384 * (size_t)n)) != cudaSuccess ||
      (e = cudaMalloc(&dLits, litBytes)) != cudaSuccess || (e = cudaMalloc(&dBuf, bufBytes)) != cudaSuccess)
    goto done;
  if ((e = cudaMemcpy(dDesc, desc, 32 * (size_t)n, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(dRuns, runs, 384 * (size_t)n, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(dLits, lits, litBytes, cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(dBuf, buf, bufBytes, cudaMemcpyHostToDevice)) != cudaSuccess)
    goto done;
  k_exec_copy<<<n < 1024 ? n : 1024, 32>>>(n, dDesc, dRuns, dLits, dBuf);
  if ((e = cudaGetLastError()) != cudaSuccess || (e = cudaDeviceSynchronize()) != cudaSuccess) goto done;
  e = cudaMemcpy(buf, dBuf, bufBytes, cudaMemcpyDeviceToHost);
done:
  cudaFree(dDesc); cudaFree(dRuns); cudaFree(dLits); cudaFree(dBuf);
  return (int)e;
}
