// zb_common.cuh — shared definitions for the libzstdb200 device code.
//
// Everything here is __host__ __device__ so that the per-thread parsers can also be compiled by g++ into
// the host simulator used by the CPU-side tests (tests/hostsim/); the product only ever runs them on the GPU.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define ZB_HD __host__ __device__ __forceinline__
#define ZB_D __device__ __forceinline__
#else
#define ZB_HD inline
#define ZB_D inline
#endif

namespace zb {

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int32_t i32;
typedef int64_t i64;
typedef int16_t s16;

// ---- result / error encoding: identical to the reference (csharp/src/ZStdErrors.cs:61-100) ----
enum : u32 {
  ZE_GENERIC = 1, ZE_prefix_unknown = 10, ZE_frameParameter_unsupported = 14, ZE_frameParameter_windowTooLarge = 16,
  ZE_corruption_detected = 20, ZE_checksum_wrong = 22, ZE_dictionary_corrupted = 30, ZE_dictionary_wrong = 32,
  ZE_tableLog_tooLarge = 44, ZE_maxSymbolValue_tooLarge = 46, ZE_maxSymbolValue_tooSmall = 48,
  ZE_workSpace_tooSmall = 66, ZE_dstSize_tooSmall = 70, ZE_srcSize_wrong = 72, ZE_maxCode = 120,
  ZB_TABLE_TOO_LARGE = 0xFFF0   // internal, never a result: a sequence table does not fit the space of this kernel instantiation
};
ZB_HD u32 zerr(u32 code) { return 0u - code; }
ZB_HD bool is_err(u32 r) { return r > zerr(ZE_maxCode); }

// ---- format constants (csharp/src/ZStd.cs:386-416,1387-1389; ZStdInternal.cs:109-209) ----
static const u32 MAGIC = 0xFD2FB528u, MAGIC_SKIP = 0x184D2A50u;
static const u32 BLOCKSIZE_MAX = 1u << 17;
static const u32 LONGNBSEQ = 0x7F00;
static const u32 MaxLL = 35, MaxML = 52, MaxOff = 31, LLFSELog = 9, MLFSELog = 9, OffFSELog = 8;
static const u32 HUF_LOG_MAX = 12;        // largest table log the reference accepts (HufDecompress.cs:128)
static const u32 HUF_TABLE_LOG = 11;      // log of the full decode table (log-12 tables are folded, zb_format.cuh)
static const u32 HUF_ROOT_SMALL = 9;      // log of the root table the Huffman kernel for small frames keeps in shared memory (zb_format.cuh huf_fill_root)
static const u32 HUF_LONG = 0xFF00u;      // root cell: the codes under this prefix are longer than the root log, look in the full table

// ---- per-item record produced by the parse kernel and refined by later stages ----
// huf_err_code value: the block's Huffman streams are well formed but its literals do not fit the frame's literal
// scratch (the output cannot fit either): the execute stage replays the block's checks without copying.
#define HUF_DRY 0xFFFFu
enum : u32 { FI_CHECKSUM = 1, FI_FCS_KNOWN = 2, FI_DONE = 4 /* result[] already final, later stages skip the item */,
              FI_NEED_XXH = 8 /* set by the execute stage: verify the content checksum */,
              FI_SMALLHUF = 32 /* few literals: its Huffman table log is at most HUF_ROOT_SMALL with any known encoder: decoded by k_huf<HUF_ROOT_SMALL> */,
              FI_SEQ_A = 64, FI_SEQ_B = 128 /* few sequences in the first block: sequence tables of at most 2^6 / 2^8 cells with any known
                                               encoder: decoded by the k_seq instantiation with tables of that size (more frames per SM) */,
              FI_PAR = 16 /* multi-block frame decoded block-parallel: its compressed blocks are BlockUnits (zb_blocks.cuh) */ };
struct FrameInfo {
  u32 flags;
  u32 body_off;      // offset within the item of the first block header of its data frame
  u64 fcs;           // frame content size when FI_FCS_KNOWN
  u64 window;        // window size (== fcs for single-segment frames)
  // entropy-stage error records (first failing block of each stage; 0xFFFFFFFF = none)
  u32 huf_err_block, huf_err_code;
  u32 seq_err_block, seq_err_code, seq_err_index;   // seq_err_index: sequences decoded before the failure; 0xFFFFFFFF = header error
  // set by the execute stage for the checksum stage
  u32 trailer_off;   // offset of the 4-byte checksum within the item
  u32 decoded;       // bytes produced by this data frame
  // items holding several data frames (DecompressMultiFrame, ZStdDecompress.cs:2096-2160) take one pass per frame
  u32 out_base;      // bytes produced by the item's earlier data frames: this frame writes at dst + out_base
  u32 next_off;      // offset within the item of the next data frame's magic (0 = none), set by the execute stage
  // FI_PAR frames: their compressed blocks are units [unit_base, unit_base + unit_count) of the slice's unit list
  u32 unit_base, unit_count;
};

// array view with a stride (bank-interleaved per-lane arrays in shared memory)
template <class T> struct Strided {
  T* p; u32 s;
  ZB_HD T& operator[](u32 i) const { return p[i * s]; }
};

// Pulls a global-memory line towards the SM ahead of a dependent load (no-op on the host simulator).
ZB_HD void prefetch_line(const void* p) {
#if defined(__CUDA_ARCH__)
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#else
  (void)p;
#endif
}

// ---- unaligned little-endian loads ----
ZB_HD u32 ld16(const u8* p) { return (u32)p[0] | ((u32)p[1] << 8); }
ZB_HD u32 ld24(const u8* p) { return (u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16); }
ZB_HD u32 ld32(const u8* p) { return (u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16) | ((u32)p[3] << 24); }
ZB_HD u64 ld64(const u8* p) { return (u64)ld32(p) | ((u64)ld32(p + 4) << 32); }

ZB_HD u32 highbit(u32 v) {   // floor(log2(v)), v != 0 (csharp/src/BitStream.cs:205-215)
#if defined(__CUDA_ARCH__)
  u32 r; asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(v)); return r;   // one FLO; 31 - __clz(v) leaves two subtractions behind
#else
  return 31 - __builtin_clz(v);
#endif
}
ZB_HD u32 fshr(u32 lo, u32 hi, u32 s) {   // low 32 bits of (hi:lo) >> (s & 31)
#if defined(__CUDA_ARCH__)
  return __funnelshift_r(lo, hi, s);
#else
  s &= 31; return s ? (lo >> s) | (hi << (32 - s)) : lo;
#endif
}

ZB_HD u32 fshl(u32 lo, u32 hi, u32 s) {   // high 32 bits of (hi:lo) << (s & 31)
#if defined(__CUDA_ARCH__)
  return __funnelshift_l(lo, hi, s);
#else
  s &= 31; return s ? (hi << s) | (lo >> (32 - s)) : hi;
#endif
}
// the top n bits of w (n < 32), and w moves past them: one 32 x 32 -> 64-bit multiplication by 2^n (an FMA-pipe
// IMAD.WIDE) in place of a subtraction and two shifts on the ALU pipe
ZB_HD u32 take_bits(u32& w, u32 n) {
  const u64 p = (u64)w * (1u << n);
  w = (u32)p;
  return (u32)(p >> 32);
}
ZB_HD u32 shr_c(u32 x, u32 n) {   // x >> n with n clamped to 32 (so n == 32 yields 0), as PTX shr.b32 defines it
#if defined(__CUDA_ARCH__)
  u32 r; asm("shr.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n)); return r;
#else
  return n >= 32 ? 0 : x >> n;
#endif
}

// ---- backward bit cursor -------------------------------------------------------------------------
// A zstd bitstream of n bytes is read from its last byte towards its first (csharp/src/BitStream.cs:322-497).
// We address it by P = number of still-unread bits counted from the first byte; reading k bits takes stream
// bits [P-k, P) and leaves P-k.  Bits below 0 read as zero (the reference's container shifts zeros in) and a
// negative P is the reference's "overflow" status.  Loads are 4-byte aligned words relative to `words`.
struct BitCursor {
  const u32* words;   // 4-byte aligned address at or below the first stream byte
  i32 gofs;           // bit offset of stream bit 0 relative to words[0] (0, 8, 16 or 24)
  i32 P;              // unread bits
};

// initialise from (src, n); returns false if n == 0 or the final byte has no end mark (BitStream.cs:324-339, 369-372)
ZB_HD bool bc_init(BitCursor& c, const u8* src, u32 n) {
  if (n < 1) return false;
  u8 last = src[n - 1];
  if (last == 0) return false;
  uintptr_t a = (uintptr_t)src;
  c.words = (const u32*)(a & ~(uintptr_t)3);
  c.gofs = (i32)(a & 3) * 8;
  c.P = (i32)(n * 8) - (i32)(8 - highbit(last));
  return true;
}

// 64 stream bits ending at P, left aligned: bit 63 of the result is stream bit P-1.  Bits below stream bit 0
// are zero.  Requires P >= 0 for meaningful data; for P < 64 only the aligned words that hold unread stream bits
// are dereferenced (nothing below `words`, nothing past the word of the last unread bit).
ZB_HD u64 bc_window64(const BitCursor& c, i32 P) {
  if (P >= 64) {
    i32 g = c.gofs + P - 64;          // bit offset (>= 0) of the window's lowest bit
    const u32* w = c.words + (g >> 5);
    u32 s = (u32)g & 31;
    u32 w0 = w[0], w1 = w[1], w2 = s ? w[2] : 0;
    u32 lo = fshr(w0, w1, s), hi = fshr(w1, w2, s);
    return ((u64)hi << 32) | lo;
  }
  if (P <= 0) return 0;
  // tail: stream bits [0, P) sit in words[0..2] from bit gofs up; only words that hold one of them are loaded
  const u32 top = (u32)c.gofs + (u32)P;                       // 1 .. 87
  const u32 w0 = c.words[0], w1 = top > 32 ? c.words[1] : 0, w2 = top > 64 ? c.words[2] : 0;
  const u32 lo = fshr(w0, w1, (u32)c.gofs), hi = fshr(w1, w2, (u32)c.gofs);
  return (((u64)hi << 32) | lo) << (64 - P);                  // bits at and above P (end mark, padding) fall off the top
}

// ---- per-thread read-ahead of a backward bitstream through shared memory ---------------------------
// Every lane of the entropy kernels walks its own bitstream, so its loads can never coalesce with its
// neighbours', and L1 is sectored: read straight from global memory nearly every step waits on an L2/HBM
// sector.  BitRing keeps the 256 bytes at and below the cursor in a per-lane ring of 16 chunks of 16 bytes in
// shared memory, filled by cp.async (LDGSTS: global -> shared without a register, so no lane's refill can stall
// another lane's use through the warp-wide register scoreboard).  A chunk is requested 13 chunks ahead of its
// first use; one commit group per step and `wait_group 12` make it certain to have landed by then.
#define ZB_RING_WORDS 64          // 16 chunks x 4 words, per lane, contiguous and 16-byte aligned
#define ZB_RING_AHEAD 13

struct BitRing {
  u32* ring;             // this lane's 64-word ring
  const u8* base16;      // 16-byte aligned address at or below the first stream byte
  i32 gofs;              // bit offset of stream bit 0 relative to base16 (0..120)
  i32 lowChunk;          // ring holds chunks lowChunk .. lowChunk+15 (chunk k = bytes [16k, 16k+16) from base16)
};

ZB_HD void ring_request(const BitRing& r, i32 chunk) {   // asynchronous on the device
  if (chunk < 0) return;                                 // below the stream: never read as data
  u32* dst = r.ring + (((u32)chunk & 15) << 2);
  const u8* src = r.base16 + (size_t)chunk * 16;
#if defined(__CUDA_ARCH__)
  const u32 saddr = (u32)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(src) : "memory");
#else
  memcpy(dst, src, 16);
#endif
}
ZB_HD void ring_commit() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.commit_group;" ::: "memory");
#endif
}
ZB_HD void ring_wait_steady() {   // all but the 12 most recent groups have landed
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.wait_group 12;" ::: "memory");
#endif
}
ZB_HD void ring_wait_all() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.wait_all;" ::: "memory");
#endif
}
// Prepares the ring for the stream src[0..nbytes).  Only valid when the cursor starts at P >= 128.
ZB_HD void ring_init(BitRing& r, u32* ring, const u8* src, u32 nbytes) {
  const uintptr_t a = (uintptr_t)src;
  r.ring = ring;
  r.base16 = (const u8*)(a & ~(uintptr_t)15);
  r.gofs = (i32)(a & 15) * 8;
  const i32 ctop = (r.gofs + (i32)nbytes * 8 - 1) >> 7;
  r.lowChunk = ctop - 15;
  for (i32 k = 0; k < 16; k++) ring_request(r, r.lowChunk + k);
  ring_commit();
  ring_wait_all();
}
// 64 stream bits ending at P (P >= 128): lo = bits [P-64, P-32), hi = [P-32, P)
ZB_HD void ring_window(const BitRing& r, i32 P, u32& lo, u32& hi) {
  ring_wait_steady();
  const i32 g = r.gofs + P - 64;
  const u32 wi = (u32)(g >> 5), sh = (u32)g & 31;
  const u32 w0 = r.ring[wi & 63], w1 = r.ring[(wi + 1) & 63], w2 = r.ring[(wi + 2) & 63];
  lo = fshr(w0, w1, sh); hi = fshr(w1, w2, sh);   // sh == 0 ignores w2
}
// Call once per step after the cursor moved to Pn (by fewer than 128 bits): keeps the ring ZB_RING_AHEAD chunks
// ahead of the window and closes this step's commit group.
// Branch-free on the device (the refill is a predicated cp.async): branches are what the one-warp-per-scheduler
// entropy loops pay most for.
ZB_HD void ring_advance(BitRing& r, i32 Pn) {
  const i32 wc = (r.gofs + Pn - 64) >> 7;
#if defined(__CUDA_ARCH__)
  const i32 chunk = r.lowChunk - 1;
  const u32 move = r.lowChunk > wc - ZB_RING_AHEAD, fetch = move && chunk >= 0;   // chunks below 0 lie before the stream
  const u32 saddr = (u32)__cvta_generic_to_shared(r.ring) + ((((u32)chunk) & 15) << 4);
  const u8* src = r.base16 + (i64)chunk * 16;
  asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p cp.async.ca.shared.global [%0], [%1], 16; }" ::"r"(saddr), "l"(src), "r"(fetch) : "memory");
  r.lowChunk -= (i32)move;
#else
  if (r.lowChunk > wc - ZB_RING_AHEAD) { r.lowChunk -= 1; ring_request(r, r.lowChunk); }
#endif
  ring_commit();
}

}  // namespace zb
