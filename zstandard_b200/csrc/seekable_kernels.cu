// seekable_kernels.cu — the device steps of seekable archives (format: seekable.h; host side: api.cu *_seekable*).
//
//   k_seek_scan  : 1 CTA          exclusive scan of the frame sizes of an encode, the table's header and footer, *dst_size
//   k_seek_pack  : warp / frame   frame from its 16-byte aligned encoder slot to its packed offset; its table entry
//   k_seek_check : warp / frame   decoded size and checksum against the table entry; first error in archive order
#include "seekable_kernels.cuh"
#include "seekable.h"
#include "xxh_device.cuh"

namespace zb {

constexpr u32 kScanThreads = 1024;
constexpr u32 kPackWarps = 8;
constexpr u64 kPackFailed = ~0ull;

// One CTA is enough: n <= max_items (65 536 for contexts up to 64 MiB), i.e. at most 64 sizes per thread, read once.
__global__ void __launch_bounds__(kScanThreads) k_seek_scan(SeekPackArgs a) {
  __shared__ u64 part[kScanThreads];
  const u32 t = threadIdx.x, per = (a.n + kScanThreads - 1) / kScanThreads;
  const u32 lo = min(a.n, t * per), hi = min(a.n, lo + per);
  u64 sum = 0; int bad = 0;
  for (u32 i = lo; i < hi; i++) { const u32 r = a.result[i]; bad |= is_err(r); sum += r; }
  bad = __syncthreads_or(bad);
  part[t] = sum;
  __syncthreads();
  for (u32 d = 1; d < kScanThreads; d <<= 1) {   // Hillis-Steele over the per-thread sums
    const u64 v = t >= d ? part[t - d] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  u64 off = part[t] - sum;
  for (u32 i = lo; i < hi; i++) { a.offsets[i] = off; off += a.result[i]; }
  if (t != kScanThreads - 1) return;
  const u64 total = part[t];
  a.offsets[a.n] = bad ? kPackFailed : total;
  if (!a.table) return;
  if (bad) { *a.dst_size = 0; return; }
  const bool ck = a.checksum != 0;
  seek::write_header(a.out + total, a.n, ck);
  seek::write_footer(a.out + total + seek::HEADER_BYTES + (u64)a.n * seek::entry_bytes(ck), a.n, ck);
  *a.dst_size = total + seek::table_bytes(a.n, ck);
}

__device__ __forceinline__ u32 sel4(u32 q, u32 a, u32 b, u32 c, u32 d) { return q == 0 ? a : (q == 1 ? b : (q == 2 ? c : d)); }

// 16 bytes starting m bytes into the 32 bytes lo:hi (m < 16), without a dynamically indexed array
__device__ __forceinline__ uint4 shifted16(uint4 lo, uint4 hi, u32 m) {
  const u32 q = m >> 2, sh = (m & 3) * 8;
  const u32 t0 = sel4(q, lo.x, lo.y, lo.z, lo.w), t1 = sel4(q, lo.y, lo.z, lo.w, hi.x), t2 = sel4(q, lo.z, lo.w, hi.x, hi.y),
            t3 = sel4(q, lo.w, hi.x, hi.y, hi.z), t4 = sel4(q, hi.x, hi.y, hi.z, hi.w);
  return make_uint4(__funnelshift_r(t0, t1, sh), __funnelshift_r(t1, t2, sh), __funnelshift_r(t2, t3, sh), __funnelshift_r(t3, t4, sh));
}

// Frame i moves from its aligned slot to out + offsets[i], an arbitrary address.  The destination's 16-byte words that the
// frame covers whole are written with one vector store each, built from two aligned source loads; the up to 15 bytes at
// either end (which share a word with the neighbouring frames, written by other warps) are written byte by byte.
__global__ void __launch_bounds__(kPackWarps * 32) k_seek_pack(SeekPackArgs a) {
  const u32 lane = threadIdx.x & 31, i = blockIdx.x * kPackWarps + (threadIdx.x >> 5);
  if (i >= a.n || a.offsets[a.n] == kPackFailed) return;
  const u32 len = a.result[i];
  const u8* s = a.frames + a.frame_off[i];
  u8* d = a.out + a.offsets[i];
  const uintptr_t d0 = (uintptr_t)d, e = d0 + len;
  uintptr_t A = (d0 + 15) & ~(uintptr_t)15, B = e & ~(uintptr_t)15;
  if (A > B) A = B = e;                                  // no whole word: all bytes go singly
  for (uintptr_t p = d0 + lane; p < A; p += 32) *(u8*)p = s[p - d0];
  for (uintptr_t p = B + lane; p < e; p += 32) *(u8*)p = s[p - d0];
  const u32 m = (u32)((A - d0) & 15);                   // source offset of word w is (A - d0) + 16 w; its misalignment is m
  const uint4* sw = (const uint4*)(s + ((A - d0) & ~(uintptr_t)15));
  const u32 words = (u32)((B - A) >> 4);
  for (u32 w = lane; w < words; w += 32) {
    const uint4 lo = sw[w];
    *(uint4*)(A + 16ull * w) = m ? shifted16(lo, sw[w + 1], m) : lo;   // sw[w + 1] stays inside the slot's aligned span
  }
  if (!a.table || lane != 0) return;
  const bool ck = a.checksum != 0;
  const u8* tail = s + len - 4;                           // every frame of a checksummed encode ends in its 4-byte checksum
  const u32 sum = ck ? ((u32)tail[0] | ((u32)tail[1] << 8) | ((u32)tail[2] << 16) | ((u32)tail[3] << 24)) : 0;
  seek::write_entry(a.out + a.offsets[a.n] + seek::HEADER_BYTES + (u64)i * seek::entry_bytes(ck), len, a.content[i], sum, ck);
}

__global__ void __launch_bounds__(SEEK_CHECK_WARPS * 32) k_seek_check(SeekCheckArgs a) {
  const u32 lane = threadIdx.x & 31, i = blockIdx.x * SEEK_CHECK_WARPS + (threadIdx.x >> 5);
  if (i < a.n) {
    const Items& it = a.it;
    u32 r = it.result[i];
    if (r == zerr(ZE_dstSize_tooSmall)) r = zerr(ZE_corruption_detected);   // capacity == the entry's size: the frame is larger
    else if (!is_err(r) && (r != it.dstCap[i] || a.info[i].next_off)) r = zerr(ZE_corruption_detected);   // one entry, one frame
    else if (!is_err(r) && a.cksum) {
      // a frame with its own checksum: the decoder has checked the trailer at trailer_off against the content, so that
      // trailer stands for it
      const FrameInfo& fi = a.info[i];
      const bool own = (fi.flags & FI_CHECKSUM) != 0;
      u32 got = 0;
      if (own) got = ld32(it.src + it.srcOff[i] + fi.trailer_off);
      else if (lane < 4) got = (u32)xxh64_group<true>(it.dst + it.dstOff[i], r, lane, 0xFu, 0);
      if (got != a.cksum[i]) r = zerr(ZE_checksum_wrong);
    }
    if (lane == 0) {
      it.result[i] = r;
      if (a.first && is_err(r)) atomicMin(a.first, ((unsigned long long)a.frame[i] << 32) | r);
    }
  }
  if (!a.code) return;
  // the last block of all check launches turns the first error into the call's code
  __syncthreads();
  if (threadIdx.x != 0) return;
  __threadfence();
  if (atomicAdd(a.done, 1u) != a.blocks_total - 1) return;
  const unsigned long long f = atomicAdd(a.first, 0ull);
  *a.code = f == ~0ull ? a.preset : (u32)f;
}

cudaError_t seek_pack(const SeekPackArgs& a, cudaStream_t st, int* launches) {
  k_seek_scan<<<1, kScanThreads, 0, st>>>(a);
  ++*launches;
  if (a.n) { k_seek_pack<<<(a.n + kPackWarps - 1) / kPackWarps, kPackWarps * 32, 0, st>>>(a); ++*launches; }
  return cudaGetLastError();
}

cudaError_t seek_check(const SeekCheckArgs& a, cudaStream_t st, int* launches) {
  k_seek_check<<<seek_check_blocks(a.n), SEEK_CHECK_WARPS * 32, 0, st>>>(a);
  ++*launches;
  return cudaGetLastError();
}

}  // namespace zb
