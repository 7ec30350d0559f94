// api.cu — host side of libzstdb200: contexts, device arenas, staging, sharding, the C ABI of include/zstdb200.h.
//
// Host responsibilities (SURVEY.md §3.4): build flat descriptor tables, shard items over the context's GPUs by
// bytes (no collective: frames are independent, ZStdDecompress.cs:2478-2499 resets all state per frame), move
// bytes host<->device and launch the kernels.  No decoding or encoding arithmetic happens on the host.
//
// Data movement.  A batch is cut into sub-batches that fit the device arenas; a sub-batch is cut into slices that
// are dealt round-robin to NSTREAMS streams, so the H2D copy of one slice, the kernels of another and the D2H
// copy of a third overlap.  When the caller's buffers are already laid out back to back (the layout a managed host gets
// from one pinned array plus offsets) they are DMA'd directly; otherwise items are gathered/scattered through the
// context's pinned staging.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/zstdb200.h"
#include "decode_kernels.cuh"
#include "dict_train.cuh"
#include "encode_kernels.cuh"
#include "zb_encode.cuh"

using namespace zb;

namespace {

constexpr int NSTREAMS = 8;
static_assert(NSTREAMS <= ENC_STREAM_PARTS, "one encoder slot partition per stream");
constexpr size_t SLICE_BYTES_DEFAULT = 32u << 20;   // uncompressed bytes per slice (several slices per stream per GiB)
constexpr size_t MIN_SLICE_ITEMS_DECODE = 1024;      // and at least this many frames (decode kernels: one frame-time per launch)
constexpr size_t MIN_SLICE_ITEMS_ENCODE = 512;       // the match kernel fills the GPU with 2-4 thousand frames: start early

// tuning aids (not part of the ABI): ZSTDB200_STREAMS = streams actually used (1..NSTREAMS), ZSTDB200_SLICE_MB
int env_int(const char* name, int dflt, int lo, int hi) {
  const char* v = getenv(name);
  if (!v || !*v) return dflt;
  int x = atoi(v);
  return x < lo ? lo : (x > hi ? hi : x);
}

struct Device {
  int id = 0;
  cudaStream_t stream[NSTREAMS] = {};
  cudaEvent_t descEv = nullptr;                 // descriptors of the current sub-batch are on the device
  std::vector<cudaEvent_t> sliceEv;             // "this slice's output is in the pinned staging" (grown on demand)
  // device memory
  u8 *d_src = nullptr, *d_dst = nullptr;       // staging for the host-pointer API
  // descriptors of one sub-batch of m items, packed so that they travel in ONE copy: [srcOff m x 8][dstOff m x 8][srcSize m x 4][dstCap m x 4]
  u8* d_desc = nullptr;
  // counters and results come back in ONE copy: [more NSTREAMS x 4][result maxItems x 4]
  u32 *d_result = nullptr;
  FrameInfo* d_info = nullptr; u8* d_lit = nullptr; SeqRec* d_seq = nullptr;
  u32* d_more = nullptr;                        // per-stream counters of items with another data frame to decode (DecodeArgs::more)
  BlockUnit* d_units = nullptr; u32* d_parList = nullptr; u32* d_cnt = nullptr;   // block-parallel path of multi-block frames (DecodeArgs::units / par_list / cnt, 2 counters per stream)
  u8* d_hufFull = nullptr; size_t hufFullBytes = 0;   // full Huffman tables of the resident frames (DecodeArgs::huf_full), one region per stream
  u8* d_dict = nullptr; size_t dictCap = 0; DictState* d_dictState = nullptr; bool dictOn = false;   // zstdb200_load_dictionary
  u8* d_encDict = nullptr; size_t encDictCap = 0;   // the same dictionary prepared for the encoder (EncDict block, zb_encode.cuh)
  EncodeScratch enc;                            // encoder arenas (encode_kernels.cuh)
  // pinned host memory
  u8 *h_src = nullptr, *h_dst = nullptr;
  u8* h_desc = nullptr;
  u64 *h_srcOff = nullptr, *h_dstOff = nullptr; u32 *h_srcSize = nullptr, *h_dstCap = nullptr;   // views into h_desc for the current sub-batch
  u32 *h_result = nullptr, *h_more = nullptr;
};

}  // namespace

struct zstdb200_ctx {
  std::vector<Device> dev;
  size_t maxBatch = 0, maxItems = 0, srcCap = 0, dstSpan = 0;
  std::string err;
  uint64_t launches = 0;
  std::vector<uint4> encDict;   // host copy of the encoder's dictionary block (enc_dict_prepare); empty: no dictionary loaded
};

namespace {

// Events of the *_timed entry points; destroyed on every return path.
template <int N> struct EventSet {
  cudaEvent_t ev[N] = {};
  ~EventSet() { for (auto e : ev) if (e) cudaEventDestroy(e); }
  cudaError_t create() { for (auto& e : ev) { cudaError_t r = cudaEventCreate(&e); if (r != cudaSuccess) return r; } return cudaSuccess; }
};

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      char b_[512]; snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      ctx->err = b_; return 1;                                                                     \
    }                                                                                              \
  } while (0)

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int alloc_device(zstdb200_ctx* ctx, Device& d) {
  CK(cudaSetDevice(d.id));
  for (auto& s : d.stream) CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&d.descEv, cudaEventDisableTiming));
  const size_t items = ctx->maxItems;
  // d_src / d_dst are the codec's input / output staging in both directions: compressed frames of a full batch can
  // be larger than the batch (compress bounds), so both buffers take the larger size
  CK(cudaMalloc(&d.d_src, ctx->srcCap + 256));
  CK(cudaMalloc(&d.d_dst, ctx->srcCap + 256));
  CK(cudaMalloc(&d.d_desc, items * 24 + 64));
  CK(cudaMalloc(&d.d_more, (NSTREAMS + items) * 4)); d.d_result = d.d_more + NSTREAMS;
  CK(cudaMallocHost(&d.h_more, (NSTREAMS + items) * 4)); d.h_result = d.h_more + NSTREAMS;
  CK(cudaMalloc(&d.d_info, items * sizeof(FrameInfo)));
  CK(cudaMalloc(&d.d_lit, decode_lit_arena_bytes(ctx->dstSpan, items)));
  CK(cudaMalloc(&d.d_seq, decode_seq_arena_bytes(ctx->dstSpan, items)));
  CK(cudaMalloc(&d.d_units, decode_unit_arena_count(ctx->dstSpan, items) * sizeof(BlockUnit)));
  CK(cudaMalloc(&d.d_parList, 4 * (items + 1) * 4));
  CK(cudaMalloc(&d.d_cnt, NSTREAMS * 8 * 4));
  CK(decode_configure());
  d.hufFullBytes = align_up(decode_huf_full_bytes(decode_huf_ctas()), 256);
  CK(cudaMalloc(&d.d_hufFull, d.hufFullBytes * NSTREAMS));
  CK(cudaMallocHost(&d.h_src, ctx->srcCap + 256)); CK(cudaMallocHost(&d.h_dst, ctx->srcCap + 256));
  CK(cudaMallocHost(&d.h_desc, items * 24 + 64));
  CK(decode_configure());
  cudaError_t ee = encode_alloc(d.enc, ctx->maxBatch, items);
  if (ee != cudaSuccess) { ctx->err = std::string("encoder arena allocation failed: ") + cudaGetErrorString(ee); return 1; }
  return 0;
}

void free_device(Device& d) {
  cudaSetDevice(d.id);
  for (auto& s : d.stream) if (s) cudaStreamSynchronize(s);
  cudaFree(d.d_src); cudaFree(d.d_dst); cudaFree(d.d_desc);
  cudaFree(d.d_info); cudaFree(d.d_lit); cudaFree(d.d_seq); cudaFree(d.d_more); cudaFreeHost(d.h_more);
  cudaFree(d.d_units); cudaFree(d.d_parList); cudaFree(d.d_cnt); cudaFree(d.d_hufFull);
  cudaFree(d.d_dict); cudaFree(d.d_dictState); cudaFree(d.d_encDict);
  encode_free(d.enc);
  cudaFreeHost(d.h_src); cudaFreeHost(d.h_dst); cudaFreeHost(d.h_desc);
  for (auto& s : d.stream) if (s) cudaStreamDestroy(s);
  if (d.descEv) cudaEventDestroy(d.descEv);
  for (auto& ev : d.sliceEv) cudaEventDestroy(ev);
}

struct Range { size_t lo, hi; };

// true when the driver can DMA the range directly (cudaMallocHost / cudaHostRegister memory).  A managed caller's
// `fixed`-pinned byte[] (ZStdDecompress.cs:2182-2186) is pinned for the GC only: pageable for CUDA.
bool is_dma_able(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// fn(lo, hi) over [0, n) on up to `maxThreads` host threads (staging copies between pageable caller memory and the
// context's pinned buffers: one thread moves ~10 GB/s, the PCIe link wants ~50)
template <class F>
void parallel_for(size_t n, size_t bytes, F fn) {
  static const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const size_t want = bytes >> 22;                                   // one thread per 4 MiB
  const size_t nt = std::min<size_t>(std::min<size_t>(hw, 16), std::min(n, want));
  if (nt <= 1) { fn(0, n); return; }
  std::vector<std::thread> th;
  for (size_t t = 0; t < nt; t++) th.emplace_back(fn, n * t / nt, n * (t + 1) / nt);
  for (auto& t : th) t.join();
}

// Sum of the frame content sizes of an item when every data frame declares one (header walk only: frame headers,
// block headers, checksum fields — ZStdDecompress.cs:2096-2160, 2033-2067).  false = unknown / malformed.
bool host_item_content_size(const u8* src, u32 size, u64* total) {
  u32 pos = 0; u64 sum = 0;
  while (true) {
    FrameInfo fi; u32 r = 0;
    if (!parse_item(src, size, fi, &r, pos, 0)) { if (is_err(r)) return false; *total = sum; return true; }
    if (!(fi.flags & FI_FCS_KNOWN)) return false;
    sum += fi.fcs;
    if (sum > 0xFFFFFFFFull) return false;
    u32 p = fi.body_off;
    while (true) {
      BlockHdr bh;
      if (read_block_hdr(src + p, size - p, bh)) return false;
      p += 3 + bh.csize;
      if (bh.last) break;
    }
    if (fi.flags & FI_CHECKSUM) { if (size - p < 4) return false; p += 4; }
    pos = p;
  }
}

// Greedy split of [0, n) into consecutive sub-batches that respect the per-device arena limits.
template <class FI, class FO>
std::vector<Range> make_subbatches(size_t n, size_t maxIn, size_t maxOut, size_t maxItems, FI inBytes, FO outBytes, bool* tooBig) {
  std::vector<Range> r; size_t lo = 0; *tooBig = false;
  while (lo < n) {
    size_t in = 0, out = 0, hi = lo;
    while (hi < n && hi - lo < maxItems) {
      size_t a = align_up(inBytes(hi), 16), b = align_up(outBytes(hi), 16);   // exactly what run_subbatch lays out
      if (in + a > maxIn || out + b > maxOut) break;
      in += a; out += b; hi++;
    }
    if (hi == lo) { *tooBig = true; return r; }   // a single item exceeds the arena
    r.push_back({lo, hi}); lo = hi;
  }
  return r;
}

enum class Op { Decompress, Compress };

// Switches a launch to the block-parallel path for multi-block frames (zb_blocks.cuh); ZSTDB200_PAR=0 keeps every frame
// on the frame-serial kernels (A/B measurements).  Also hands every launch its per-stream scratch: slot = the stream slot
// the launch runs on (its eight counters, its Huffman full-table region); the item lists are indexed by item_base, so
// slices of one sub-batch that run concurrently use disjoint ranges of them.
void with_units(Device& d, DecodeArgs& a, u32 slot, size_t ctx_items) {
  static const bool on = env_int("ZSTDB200_PAR", 1, 0, 1) != 0;
  static const u32 seqAMax = (u32)env_int("ZSTDB200_SEQ_A_MAX", 512, 0, 0x7FFFFFFF), seqBMax = (u32)env_int("ZSTDB200_SEQ_B_MAX", 2048, 0, 0x7FFFFFFF);
  a.seq_a_max = seqAMax; a.seq_b_max = seqBMax;
  a.huf_full = (u16*)(d.d_hufFull + d.hufFullBytes * slot);       // (every launch: the Huffman kernels' full-table scratch and the counters of this stream)
  a.cnt = d.d_cnt + 8 * slot; a.par_list = d.d_parList; a.list_stride = (u32)(ctx_items + 1);
  if (!on) return;
  a.units = d.d_units;
}

// Items that hold more than one data frame (DecompressMultiFrame, ZStdDecompress.cs:2096-2160): after the first pass
// the execute stage has counted them in *more; every further pass decodes the next data frame of each of them.
// Synchronises `st` once per pass (the count has to reach the host).  `a` covers the same items as the first pass.
cudaError_t decode_more_passes(Device& d, DecodeArgs a, u32 slot, cudaStream_t st, int* launches) {
  cudaError_t e;
  while (true) {
    a.pass++; a.more = d.d_more + slot;
    if ((e = cudaMemsetAsync(a.more, 0, 4, st)) != cudaSuccess) return e;
    if ((e = decode_launch(a, st, launches)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(d.h_more + slot, a.more, 4, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    if (d.h_more[slot] == 0) return cudaSuccess;
  }
}

struct Job {
  Op op; int level, checksum;
  const void* const* src; const uint32_t* srcSize; void* const* dst; const uint32_t* dstCap; uint32_t* result;
  // Capacity each item gets on the device: min(dstCap, what a well-formed item can produce) — a caller's large reusable
  // scratch buffer must not reserve that much of the arenas (run_host_batch).  == dstCap unless clamped.
  const uint32_t* effCap;
  uint32_t maxSrc;     // largest srcSize of the call (compress: table sizes of the match stage)
  bool useDict;        // compress with the context's dictionary (the *_using_dict calls)
};

// The encoder's dictionary on device d (zstdb200_load_dictionary put it on every device of the context)
void set_dict(const zstdb200_ctx* ctx, const Device& d, EncodeArgs& a) {
  const EncDict* h = reinterpret_cast<const EncDict*>(ctx->encDict.data());
  a.dict = reinterpret_cast<const EncDict*>(d.d_encDict); a.dict_id = h->dictID; a.dict_err = h->err;
}

// One sub-batch [lo, hi) on one device: slices over NSTREAMS streams, direct DMA where the layout allows.
// Returns "" or an error description.
std::string run_subbatch(zstdb200_ctx* ctx, Device& d, const Job& j, size_t lo, size_t hi, uint64_t* launches) {
  const size_t m = hi - lo;
  auto fail = [&](const char* what, cudaError_t e) { return std::string(what) + ": " + cudaGetErrorString(e); };
  // ---- layout analysis ----
  bool srcDirect = true, dstDirect = true;
  for (size_t k = 0; k + 1 < m && (srcDirect || dstDirect); k++) {
    const size_t i = lo + k;
    const u8 *s0 = (const u8*)j.src[i], *s1 = (const u8*)j.src[i + 1];
    if (!(s1 >= s0 + j.srcSize[i] && s1 <= s0 + j.srcSize[i] + 64)) srcDirect = false;
    const u8 *d0 = (const u8*)j.dst[i], *d1 = (const u8*)j.dst[i + 1];
    if (d1 != d0 + j.dstCap[i] || j.effCap[i] != j.dstCap[i]) dstDirect = false;
  }
  if (j.effCap[hi - 1] != j.dstCap[hi - 1]) dstDirect = false;
  const u8* srcBase = (const u8*)j.src[lo]; u8* dstBase = (u8*)j.dst[lo];
  // pageable caller memory goes through the pinned staging with parallel host copies (a pageable cudaMemcpyAsync
  // is a synchronous, single-threaded bounce inside the driver)
  if (srcDirect && !is_dma_able(srcBase)) srcDirect = false;
  if (dstDirect && !is_dma_able(dstBase)) dstDirect = false;
  if (srcDirect) {
    const size_t span = (size_t)((const u8*)j.src[hi - 1] - srcBase) + j.srcSize[hi - 1];
    const size_t lim = j.op == Op::Decompress ? ctx->srcCap : ctx->dstSpan;
    if (span > lim || !srcBase) srcDirect = false;
  }
  if (dstDirect) {
    const size_t span = (size_t)((u8*)j.dst[hi - 1] - dstBase) + j.effCap[hi - 1];
    const size_t lim = j.op == Op::Decompress ? ctx->dstSpan : ctx->srcCap;
    if (span > lim || !dstBase) dstDirect = false;
  }
  // ---- descriptors (device offsets), packed for this m ----
  d.h_srcOff = (u64*)d.h_desc; d.h_dstOff = d.h_srcOff + m; d.h_srcSize = (u32*)(d.h_dstOff + m); d.h_dstCap = d.h_srcSize + m;
  u64* const d_srcOff = (u64*)d.d_desc; u64* const d_dstOff = d_srcOff + m; u32* const d_srcSize = (u32*)(d_dstOff + m); u32* const d_dstCap = d_srcSize + m;
  size_t in = 0, out = 0;
  for (size_t k = 0; k < m; k++) {
    const size_t i = lo + k;
    d.h_srcSize[k] = j.srcSize[i]; d.h_dstCap[k] = j.effCap[i];
    d.h_srcOff[k] = srcDirect ? (u64)((const u8*)j.src[i] - srcBase) : in;
    d.h_dstOff[k] = dstDirect ? (u64)((u8*)j.dst[i] - dstBase) : out;
    in += align_up(j.srcSize[i], 16); out += align_up(j.effCap[i], 16);
  }
  // ---- slices ----
  static const int nStreams = env_int("ZSTDB200_STREAMS", NSTREAMS, 1, NSTREAMS);
  static const size_t SLICE_BYTES = (size_t)env_int("ZSTDB200_SLICE_MB", (int)(SLICE_BYTES_DEFAULT >> 20), 1, 4096) << 20;
  std::vector<Range> slices;
  {
    size_t a = 0;
    while (a < m) {
      size_t b = a, bytes = 0;
      // a slice is >= SLICE_BYTES and >= MIN_SLICE_ITEMS frames: the kernels take one frame-time however few frames
      // they are given, so slices of a few large frames would serialise on that latency
      static const int envMin = env_int("ZSTDB200_MIN_SLICE_ITEMS", 0, 0, 1 << 30);
      const size_t minItems = envMin ? (size_t)envMin : (j.op == Op::Decompress ? MIN_SLICE_ITEMS_DECODE : MIN_SLICE_ITEMS_ENCODE);
      // The first slices are smaller: output can only start to leave once a slice's kernels are done (one frame-time
      // however small the slice), and the D2H engine then has to be fed without a gap while the big slices finish.
      const size_t k = slices.size(), shrink = j.op == Op::Decompress ? (k < 2 ? 4 : (k < 4 ? 2 : 1)) : 1;
      const size_t wantItems = std::max<size_t>(1, minItems / shrink), wantBytes = SLICE_BYTES / shrink;
      while (b < m && (b - a < wantItems || bytes + std::max(d.h_dstCap[b], d.h_srcSize[b]) <= wantBytes)) { bytes += std::max(d.h_dstCap[b], d.h_srcSize[b]); b++; }
      slices.push_back({a, b}); a = b;
    }
  }
  cudaError_t e;
  // Small copies cost the copy engines about as much as a megabyte each, and they queue between the slices'
  // payload copies: descriptors go up once per sub-batch, results and counters come back once at its end.
  {
    cudaStream_t s0 = d.stream[0];
    e = cudaMemsetAsync(d.d_more, 0, NSTREAMS * 4, s0); if (e) return fail("memset", e);
    e = cudaMemcpyAsync(d.d_desc, d.h_desc, m * 24, cudaMemcpyHostToDevice, s0); if (e) return fail("H2D desc", e);
    if (slices.size() > 1) {
      e = cudaEventRecord(d.descEv, s0); if (e) return fail("event", e);
      for (int k = 1; k < NSTREAMS; k++) { e = cudaStreamWaitEvent(d.stream[k], d.descEv, 0); if (e) return fail("event wait", e); }
    }
  }
  static const bool trace = getenv("ZSTDB200_TRACE") != nullptr;   // per-slice timeline on stderr (tuning aid)
  const bool eager = !dstDirect && j.op == Op::Decompress && slices.size() > 1;
  if (eager) while (d.sliceEv.size() < slices.size()) { cudaEvent_t ev; e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming); if (e) return fail("event create", e); d.sliceEv.push_back(ev); }
  std::vector<cudaEvent_t> tev;
  if (trace) { tev.resize(1 + 3 * slices.size()); for (auto& x : tev) cudaEventCreate(&x); cudaEventRecord(tev[0], d.stream[0]); }
  for (size_t s = 0; s < slices.size(); s++) {
    const size_t a = slices[s].lo, b = slices[s].hi, cnt = b - a;
    cudaStream_t st = d.stream[s % nStreams];
    // input bytes of the slice
    const size_t inLo = d.h_srcOff[a], inHi = d.h_srcOff[b - 1] + d.h_srcSize[b - 1];
    if (srcDirect) {
      if (inHi > inLo) { e = cudaMemcpyAsync(d.d_src + inLo, srcBase + inLo, inHi - inLo, cudaMemcpyHostToDevice, st); if (e) return fail("H2D src", e); }
    } else {
      parallel_for(b - a, inHi - inLo, [&](size_t x, size_t y) {
        for (size_t k = a + x; k < a + y; k++) if (d.h_srcSize[k]) memcpy(d.h_src + d.h_srcOff[k], j.src[lo + k], d.h_srcSize[k]);
      });
      if (inHi > inLo) { e = cudaMemcpyAsync(d.d_src + inLo, d.h_src + inLo, inHi - inLo, cudaMemcpyHostToDevice, st); if (e) return fail("H2D src", e); }
    }
    if (trace) cudaEventRecord(tev[1 + 3 * s], st);
    int nl = 0;
    if (j.op == Op::Decompress) {
      DecodeArgs ar{d.d_src, d_srcOff + a, d_srcSize + a, d.d_dst, d_dstOff + a, d_dstCap + a, d.d_result + a, (u32)cnt, (u32)a,
                    d.d_info + a, d.d_lit, d.d_seq, d.dictOn ? d.d_dictState : nullptr, d.d_dict, 0, d.d_more + (s % nStreams)};
      with_units(d, ar, (u32)(s % nStreams), ctx->maxItems);
      e = decode_launch(ar, st, &nl);
    } else {
      EncodeArgs ar{d.d_src, d_srcOff + a, d_srcSize + a, d.d_dst, d_dstOff + a, d_dstCap + a, d.d_result + a, (u32)cnt, (u32)a,
                    j.level, j.checksum, j.maxSrc, (u32)(s % nStreams)};
      if (j.useDict) set_dict(ctx, d, ar);
      e = encode_launch(ar, d.enc, st, &nl);
    }
    *launches += nl;
    if (e) return fail("kernel launch", e);
    if (trace) cudaEventRecord(tev[2 + 3 * s], st);
    const size_t outLo = d.h_dstOff[a], outHi = d.h_dstOff[b - 1] + d.h_dstCap[b - 1];
    if (outHi > outLo) {
      u8* hostDst = dstDirect ? dstBase + outLo : d.h_dst + outLo;
      e = cudaMemcpyAsync(hostDst, d.d_dst + outLo, outHi - outLo, cudaMemcpyDeviceToHost, st); if (e) return fail("D2H dst", e);
    }
    if (trace) cudaEventRecord(tev[3 + 3 * s], st);
    if (eager) { e = cudaEventRecord(d.sliceEv[s], st); if (e) return fail("event", e); }
  }
  // Pageable destinations of a decode: scatter every slice out of the pinned staging as soon as its copy has landed,
  // while the later slices are still in flight (the whole capacity of each item is copied: the result codes only arrive
  // at the end; bytes past result[i] are unspecified, include/zstdb200.h).
  if (eager)
    for (size_t s = 0; s < slices.size(); s++) {
      e = cudaEventSynchronize(d.sliceEv[s]); if (e) return fail("event sync", e);
      const size_t a = slices[s].lo, b = slices[s].hi;
      parallel_for(b - a, d.h_dstOff[b - 1] + d.h_dstCap[b - 1] - d.h_dstOff[a], [&](size_t x, size_t y) {
        for (size_t k = a + x; k < a + y; k++) if (d.h_dstCap[k]) memcpy(j.dst[lo + k], d.h_dst + d.h_dstOff[k], d.h_dstCap[k]);
      });
    }
  // a single slice ran on stream 0 alone: its results ride the same stream and one synchronisation ends the call
  if (slices.size() > 1) for (auto& st : d.stream) { e = cudaStreamSynchronize(st); if (e) return fail("stream sync", e); }
  if (trace) {
    if (slices.size() == 1) cudaStreamSynchronize(d.stream[0]);
    for (size_t s = 0; s < slices.size(); s++) {
      float t1 = 0, t2 = 0, t3 = 0;
      cudaEventElapsedTime(&t1, tev[0], tev[1 + 3 * s]); cudaEventElapsedTime(&t2, tev[0], tev[2 + 3 * s]); cudaEventElapsedTime(&t3, tev[0], tev[3 + 3 * s]);
      fprintf(stderr, "[zstdb200] slice %2zu items %6zu: h2d done %7.3f  kernels done %7.3f  d2h done %7.3f ms\n", s, slices[s].hi - slices[s].lo, t1, t2, t3);
    }
    for (auto& x : tev) cudaEventDestroy(x);
  }
  e = cudaMemcpyAsync(d.h_more, d.d_more, (NSTREAMS + m) * 4, cudaMemcpyDeviceToHost, d.stream[0]); if (e) return fail("D2H results", e);
  e = cudaStreamSynchronize(d.stream[0]); if (e) return fail("stream sync", e);
  u32 anyMore = 0;
  for (int k = 0; k < NSTREAMS; k++) anyMore |= d.h_more[k];
  if (j.op == Op::Decompress && anyMore) {
    // rare path: some items hold several data frames.  Everything is still resident: decode the remaining frames
    // pass by pass over the whole sub-batch, then fetch results and output again.
    cudaStream_t st = d.stream[0]; int nl = 0;
    DecodeArgs ar{d.d_src, d_srcOff, d_srcSize, d.d_dst, d_dstOff, d_dstCap, d.d_result, (u32)m, 0, d.d_info, d.d_lit, d.d_seq, d.dictOn ? d.d_dictState : nullptr, d.d_dict, 0, nullptr};
    with_units(d, ar, 0, ctx->maxItems);
    e = decode_more_passes(d, ar, 0, st, &nl); *launches += nl;
    if (e) return fail("multi-frame passes", e);
    e = cudaMemcpyAsync(d.h_result, d.d_result, m * 4, cudaMemcpyDeviceToHost, st); if (e) return fail("D2H result", e);
    const size_t outLo = d.h_dstOff[0], outHi = d.h_dstOff[m - 1] + d.h_dstCap[m - 1];
    if (outHi > outLo) { e = cudaMemcpyAsync(dstDirect ? dstBase + outLo : d.h_dst + outLo, d.d_dst + outLo, outHi - outLo, cudaMemcpyDeviceToHost, st); if (e) return fail("D2H dst", e); }
    e = cudaStreamSynchronize(st); if (e) return fail("stream sync", e);
  }
  for (size_t k = 0; k < m; k++) j.result[lo + k] = d.h_result[k];
  // staged output not scattered yet (compress: frames are much smaller than their capacity; single-slice calls; items
  // that needed further passes): copy what was produced; on error the reference leaves dst partially written, we copy nothing
  if (!dstDirect && (!eager || anyMore)) parallel_for(m, d.h_dstOff[m - 1] + d.h_dstCap[m - 1], [&](size_t x, size_t y) {
    for (size_t k = x; k < y; k++) {
      const size_t i = lo + k; const u32 r = d.h_result[k];
      if (!is_err(r) && r) memcpy(j.dst[i], d.h_dst + d.h_dstOff[k], std::min<u32>(r, j.dstCap[i]));
    }
  });
  return "";
}

int run_host_batch(zstdb200_ctx* ctx, const Job& j0, size_t n, bool clamp = true) {
  if (n == 0) return 0;
  if (!j0.src || !j0.srcSize || !j0.dst || !j0.dstCap || !j0.result) { ctx->err = "null argument"; return 1; }
  // staging limits.  decode: in = frames (d_src, srcCap), out = content (dstSpan: what the literal / sequence arenas
  // are sized for); encode: in = raw chunks (dstSpan: what the encoder arenas are sized for), out = frames (d_dst, srcCap)
  const size_t maxIn = j0.op == Op::Decompress ? ctx->srcCap : ctx->dstSpan;
  const size_t maxOut = j0.op == Op::Decompress ? ctx->dstSpan : ctx->srcCap;
  // Device-side capacity per item.  The reference accepts any dstCapacity (a small frame into a large reusable scratch
  // buffer is fine, ZStdDecompress.cs:2182-2191), so the arenas must not be sized by it:
  //  * compress: no frame is larger than compress_bound(srcSize);
  //  * decompress: when every data frame of the item declares its content size, a well-formed item produces exactly
  //    their sum.  A malformed one may try to produce more; its dstSize_tooSmall under the clamped capacity says
  //    nothing about the caller's real one, so such items are run again below with the caller's capacity;
  //  * either way at most what the arena of a lone item holds (the limit of this context, reported as an error).
  std::vector<uint32_t> eff(n);
  const size_t lone = (maxOut & ~(size_t)15) - 16;
  for (size_t i = 0; i < n; i++) {
    uint64_t c = j0.dstCap[i];
    if (clamp) {
      if (j0.op == Op::Compress) c = std::min<uint64_t>(c, encode_bound(j0.srcSize[i]));
      else if (j0.src[i] && j0.srcSize[i] >= 5) {
        const u64 declared = zstdb200_get_decompressed_size(j0.src[i], j0.srcSize[i]);   // first frame's header only: cheap filter
        u64 total;
        if (declared && declared < c && host_item_content_size((const u8*)j0.src[i], j0.srcSize[i], &total)) c = std::min<uint64_t>(c, total);
      }
    }
    eff[i] = (uint32_t)std::min<uint64_t>(c, lone);
  }
  Job j = j0; j.effCap = eff.data();
  if (clamp) { j.maxSrc = 0; for (size_t i = 0; i < n; i++) j.maxSrc = std::max(j.maxSrc, j0.srcSize[i]); }
  bool tooBig = false;
  std::vector<Range> subs = make_subbatches(n, maxIn, maxOut, ctx->maxItems,
      [&](size_t i) { return (size_t)j.srcSize[i]; }, [&](size_t i) { return (size_t)j.effCap[i]; }, &tooBig);
  if (tooBig) { ctx->err = "an item is larger than the context's max_batch_bytes"; return 1; }
  // a single sub-batch on a multi-GPU context is re-cut so that every device gets a share
  const size_t nd = ctx->dev.size();
  if (nd > 1 && subs.size() < nd) {
    std::vector<Range> cut;
    for (auto& r : subs) {
      // equal shares of bytes (in + out), not of items: a raw-block frame costs a copy, a text frame a full decode
      const size_t parts = std::min(nd, r.hi - r.lo);
      uint64_t total = 0;
      for (size_t i = r.lo; i < r.hi; i++) total += (uint64_t)j.srcSize[i] + j.effCap[i] + 1;
      size_t lo = r.lo; uint64_t acc = 0;
      for (size_t p = 0; p < parts; p++) {
        size_t hi = lo;
        const uint64_t want = total * (p + 1) / parts;
        while (hi < r.hi && (acc < want || hi == lo) && (r.hi - hi) > (parts - 1 - p)) { acc += (uint64_t)j.srcSize[hi] + j.effCap[hi] + 1; hi++; }
        if (p + 1 == parts) hi = r.hi;
        cut.push_back({lo, hi}); lo = hi;
      }
    }
    subs.swap(cut);
  }
  std::vector<std::string> errs(nd);
  std::vector<uint64_t> launches(nd, 0);
  auto worker = [&](size_t di) {
    Device& d = ctx->dev[di];
    cudaError_t e = cudaSetDevice(d.id);
    if (e != cudaSuccess) { errs[di] = std::string("cudaSetDevice: ") + cudaGetErrorString(e); return; }
    for (size_t s = di; s < subs.size(); s += nd) {
      errs[di] = run_subbatch(ctx, d, j, subs[s].lo, subs[s].hi, &launches[di]);
      if (!errs[di].empty()) return;
    }
  };
  if (nd == 1 || subs.size() == 1) { for (size_t di = 0; di < nd; di++) worker(di); }
  else { std::vector<std::thread> th; for (size_t di = 0; di < nd; di++) th.emplace_back(worker, di); for (auto& t : th) t.join(); }
  for (size_t di = 0; di < nd; di++) ctx->launches += launches[di];
  for (size_t di = 0; di < nd; di++) if (!errs[di].empty()) { ctx->err = "device " + std::to_string(ctx->dev[di].id) + ": " + errs[di]; return 1; }
  // items that ran out of a capacity smaller than the caller's: once more with the real one (malformed frames that
  // overshoot their declared size, or items larger than what the arenas were clamped to)
  std::vector<size_t> again;
  for (size_t i = 0; i < n; i++) if (eff[i] < j.dstCap[i] && j.result[i] == zerr(ZE_dstSize_tooSmall)) again.push_back(i);
  if (!again.empty()) {
    if (!clamp) { ctx->err = "an item is larger than the context's max_batch_bytes"; return 1; }
    const size_t m = again.size();
    std::vector<const void*> s2(m); std::vector<void*> d2(m); std::vector<uint32_t> ss2(m), dc2(m), r2(m);
    for (size_t k = 0; k < m; k++) { const size_t i = again[k]; s2[k] = j.src[i]; d2[k] = j.dst[i]; ss2[k] = j.srcSize[i]; dc2[k] = j.dstCap[i]; }
    Job jr{j.op, j.level, j.checksum, s2.data(), ss2.data(), d2.data(), dc2.data(), r2.data(), nullptr, j.maxSrc, j.useDict};
    if (run_host_batch(ctx, jr, m, false)) return 1;
    for (size_t k = 0; k < m; k++) j.result[again[k]] = r2[k];
  }
  return 0;
}

}  // namespace

extern "C" {

const char* zstdb200_version(void) { return "zstdb200 0.1 (sm_100a)"; }

int zstdb200_create(zstdb200_ctx** out, const int* devices, int n_devices, size_t max_batch_bytes) {
  if (!out) return 1;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return 2;   // no CUDA device: there is no CPU fallback
  zstdb200_ctx* ctx = new zstdb200_ctx();
  if (max_batch_bytes < (1u << 20)) max_batch_bytes = 1u << 20;
  ctx->maxBatch = align_up(max_batch_bytes, 4096);
  ctx->maxItems = std::max<size_t>(65536, ctx->maxBatch / 1024);
  ctx->dstSpan = ctx->maxBatch + 16 * ctx->maxItems;
  ctx->srcCap = ctx->maxBatch + ctx->maxBatch / 128 + 128 * ctx->maxItems;   // >= sum of compress bounds of a full batch
  int one = 0;
  if (!devices || n_devices <= 0) { devices = &one; n_devices = 1; }
  for (int i = 0; i < n_devices; i++) {
    if (devices[i] < 0 || devices[i] >= count) { delete ctx; return 3; }
    Device d; d.id = devices[i]; ctx->dev.push_back(d);
  }
  for (auto& d : ctx->dev)
    if (alloc_device(ctx, d)) { fprintf(stderr, "zstdb200_create: %s\n", ctx->err.c_str()); for (auto& x : ctx->dev) free_device(x); delete ctx; return 4; }
  *out = ctx;
  return 0;
}

void zstdb200_destroy(zstdb200_ctx* ctx) {
  if (!ctx) return;
  for (auto& d : ctx->dev) free_device(d);
  delete ctx;
}

const char* zstdb200_last_error(const zstdb200_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
size_t zstdb200_max_items(const zstdb200_ctx* ctx) { return ctx ? ctx->maxItems : 0; }
int zstdb200_device_count(const zstdb200_ctx* ctx) { return ctx ? (int)ctx->dev.size() : 0; }
uint64_t zstdb200_kernel_launches(const zstdb200_ctx* ctx) { return ctx ? ctx->launches : 0; }

int zstdb200_is_error(uint32_t code) { return is_err(code); }

// Host-only frame-header parse, ZStdDecompress.cs:518-531, 590-622 (same rules as parse_item in zb_format.cuh).
uint64_t zstdb200_get_decompressed_size(const void* src, uint32_t srcSize) {
  const u8* p = (const u8*)src;
  if (!p || srcSize < 5) return 0;
  u32 magic = ld32(p);
  if (magic != MAGIC) return 0;                       // skippable frame -> 0, unknown prefix -> 0
  u32 fhd = p[4], did = fhd & 3, single = (fhd >> 5) & 1, fcsId = fhd >> 6;
  u32 fhs = 5 + (single ? 0 : 1) + (did == 3 ? 4 : did) + (fcsId == 0 ? 0 : (1u << fcsId)) + ((single && fcsId == 0) ? 1 : 0);
  if (srcSize < fhs) return 0;
  if (fhd & 0x08) return 0;
  u32 pos = 5;
  if (!single) { u32 wl = p[pos++]; if ((wl >> 3) + 10 > 30) return 0; }
  pos += did == 3 ? 4 : did;
  u64 fcs;
  if (fcsId == 0) { if (!single) return 0; fcs = p[pos]; }
  else if (fcsId == 1) fcs = ld16(p + pos) + 256;
  else if (fcsId == 2) fcs = ld32(p + pos);
  else fcs = ld64(p + pos);
  return fcs >= 0xFFFFFFFFFFFFFFFEull ? 0 : fcs;
}

// ZSTD_decompress_usingDict (ZStdDecompress.cs:2162-2167; dictionary loading :2366-2475): the dictionary becomes part of
// the context and every later decompress call starts each data frame from it.  dict == NULL or dictSize == 0 removes it.
int zstdb200_load_dictionary(zstdb200_ctx* ctx, const void* dict, uint32_t dictSize) {
  if (!ctx) return 1;
  ctx->err.clear();
  // the encoder's preparation, once on the host (the same dict_load the decoder runs in k_dict, then enc_dict_prepare);
  // every device gets a copy of the block
  ctx->encDict.clear();
  if (dict && dictSize) {
    std::vector<u8> bytes((const u8*)dict, (const u8*)dict + dictSize); bytes.resize((size_t)dictSize + 64, 0);
    std::unique_ptr<DictState> ds(new DictState());
    HufBuildWk wk; HufFseScratch fs; u8 slot[260]; s16 norm[64]; u16 next[64];
    dict_load(bytes.data(), dictSize, *ds, wk, fs, slot, norm, next);
    ctx->encDict.assign((enc_dict_bytes(ds->err ? 0 : ds->contentSize) + 15) / 16, uint4{});
    std::vector<u8> tableSymbol(512);
    enc_dict_prepare(bytes.data(), dictSize, *ds, reinterpret_cast<EncDict*>(ctx->encDict.data()), wk, fs, slot, tableSymbol.data());
  }
  for (auto& d : ctx->dev) {
    CK(cudaSetDevice(d.id));
    if (!dict || dictSize == 0) { d.dictOn = false; continue; }
    if (dictSize + 64 > d.dictCap) {
      cudaFree(d.d_dict); d.d_dict = nullptr; d.dictCap = 0;
      CK(cudaMalloc(&d.d_dict, (size_t)dictSize + 64)); d.dictCap = (size_t)dictSize + 64;
    }
    if (!d.d_dictState) CK(cudaMalloc(&d.d_dictState, sizeof(DictState)));
    CK(cudaMemcpyAsync(d.d_dict, dict, dictSize, cudaMemcpyHostToDevice, d.stream[0]));
    CK(decode_load_dictionary(d.d_dict, dictSize, d.d_dictState, d.stream[0]));
    const size_t encBytes = ctx->encDict.size() * sizeof(uint4);
    if (encBytes > d.encDictCap) {
      cudaFree(d.d_encDict); d.d_encDict = nullptr; d.encDictCap = 0;
      CK(cudaMalloc(&d.d_encDict, encBytes)); d.encDictCap = encBytes;
    }
    CK(cudaMemcpyAsync(d.d_encDict, ctx->encDict.data(), encBytes, cudaMemcpyHostToDevice, d.stream[0]));
    CK(cudaStreamSynchronize(d.stream[0]));
    d.dictOn = true;
  }
  return 0;
}

int zstdb200_decompress_batch(zstdb200_ctx* ctx, const void* const* src, const uint32_t* srcSize,
                              void* const* dst, const uint32_t* dstCap, uint32_t* result, size_t n) {
  if (!ctx) return 1;
  ctx->err.clear();
  Job j{Op::Decompress, 0, 0, src, srcSize, dst, dstCap, result, nullptr, 0, false};
  return run_host_batch(ctx, j, n);
}

uint32_t zstdb200_decompress(zstdb200_ctx* ctx, void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize) {
  uint32_t r = zerr(ZE_GENERIC);
  const void* s = src; void* d = dst;
  static unsigned char dummy[16];
  if (!d) { d = dummy; dstCapacity = 0; }        // a null array is an empty one (the C# shim passes null for byte[0])
  if (!s) { s = dummy; srcSize = 0; }
  if (zstdb200_decompress_batch(ctx, &s, &srcSize, &d, &dstCapacity, &r, 1)) return zerr(ZE_GENERIC);
  return r;
}

// Device-resident decode: one launch sequence over the whole batch on the caller's stream (slicing a resident batch
// over several streams was measured slower: whole-batch kernels fill the GPU better).  The count of items that
// hold a further data frame has to reach the host, so this entry point synchronises the stream once per pass.
static int decode_device(zstdb200_ctx* ctx, Device& d, const DecodeArgs& a, cudaStream_t user, cudaEvent_t* marks) {
  int nl = 0;
  DecodeArgs b = a; b.pass = 0; b.more = d.d_more;
  with_units(d, b, 0, ctx->maxItems);
  CK(cudaMemsetAsync(b.more, 0, 4, user));
  CK(decode_launch(b, user, &nl, marks));
  CK(cudaMemcpyAsync(d.h_more, b.more, 4, cudaMemcpyDeviceToHost, user));
  CK(cudaStreamSynchronize(user));
  if (d.h_more[0]) CK(decode_more_passes(d, b, 0, user, &nl));
  ctx->launches += nl;
  return 0;
}

int zstdb200_decompress_batch_device(zstdb200_ctx* ctx, int device_index, const void* src_base, const uint64_t* src_off,
                                     const uint32_t* src_size, void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                     uint32_t* result, size_t n, void* stream) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (device_index < 0 || device_index >= (int)ctx->dev.size()) { ctx->err = "bad device_index"; return 1; }
  if (n > ctx->maxItems) { ctx->err = "n exceeds zstdb200_max_items"; return 1; }
  Device& d = ctx->dev[device_index];
  CK(cudaSetDevice(d.id));
  DecodeArgs a{(const u8*)src_base, src_off, src_size, (u8*)dst_base, dst_off, dst_cap, result, (u32)n, 0, d.d_info, d.d_lit, d.d_seq, d.dictOn ? d.d_dictState : nullptr, d.d_dict, 0, nullptr};
  return decode_device(ctx, d, a, stream ? (cudaStream_t)stream : d.stream[0], nullptr);
}

// Same work as one launch sequence with CUDA events between the kernels: per-kernel device times for the
// bench's roofline block.
int zstdb200_decompress_batch_device_timed(zstdb200_ctx* ctx, int device_index, const void* src_base, const uint64_t* src_off,
                                           const uint32_t* src_size, void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                           uint32_t* result, size_t n, void* stream, float* kernel_ms, int max_kernels) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (device_index < 0 || device_index >= (int)ctx->dev.size()) { ctx->err = "bad device_index"; return 1; }
  if (n > ctx->maxItems) { ctx->err = "n exceeds zstdb200_max_items"; return 1; }
  Device& d = ctx->dev[device_index];
  CK(cudaSetDevice(d.id));
  cudaStream_t st = stream ? (cudaStream_t)stream : d.stream[0];
  EventSet<DECODE_KERNELS + 1> es; CK(es.create());
  cudaEvent_t* ev = es.ev;
  DecodeArgs a{(const u8*)src_base, src_off, src_size, (u8*)dst_base, dst_off, dst_cap, result, (u32)n, 0, d.d_info, d.d_lit, d.d_seq, d.dictOn ? d.d_dictState : nullptr, d.d_dict, 0, nullptr};
  if (decode_device(ctx, d, a, st, ev)) return 1;
  CK(cudaStreamSynchronize(st));
  for (int k = 0; k < DECODE_KERNELS && k < max_kernels; k++) CK(cudaEventElapsedTime(&kernel_ms[k], ev[k], ev[k + 1]));
  return 0;
}
const char* zstdb200_decode_kernel_name(int k) { return (k >= 0 && k < DECODE_KERNELS) ? kDecodeKernelNames[k] : ""; }

size_t zstdb200_compress_bound(size_t srcSize) { return encode_bound(srcSize); }

// The device-pointer compress entry points learn the largest chunk of the call (it selects the match stage's table
// sizes) by fetching the size array once: one small copy and one synchronisation of the stream.
static int device_max_u32(zstdb200_ctx* ctx, Device& d, const uint32_t* d_vals, size_t n, cudaStream_t st, u32* out) {
  *out = 0;
  if (n == 0) return 0;
  u32* h = (u32*)d.h_desc;
  CK(cudaMemcpyAsync(h, d_vals, n * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (size_t i = 0; i < n; i++) *out = std::max(*out, h[i]);
  return 0;
}

// The compress entry points with and without the context's dictionary share these bodies (useDict).
static int compress_batch(zstdb200_ctx* ctx, int level, int checksum, const void* const* src, const uint32_t* srcSize,
                          void* const* dst, const uint32_t* dstCap, uint32_t* result, size_t n, bool useDict) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (level < 1 || level > 3) { ctx->err = "level must be 1..3"; return 1; }
  if (useDict && ctx->encDict.empty()) { ctx->err = "no dictionary loaded (zstdb200_load_dictionary)"; return 1; }
  Job j{Op::Compress, level, checksum, src, srcSize, dst, dstCap, result, nullptr, 0, useDict};
  return run_host_batch(ctx, j, n);
}

static uint32_t compress_one(zstdb200_ctx* ctx, int level, int checksum, void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize,
                             bool useDict) {
  uint32_t r = zerr(ZE_GENERIC);
  const void* s = src; void* d = dst;
  static unsigned char dummy[16];
  if (!s) { s = dummy; srcSize = 0; }
  if (!d) { d = dummy; dstCapacity = 0; }
  if (compress_batch(ctx, level, checksum, &s, &srcSize, &d, &dstCapacity, &r, 1, useDict)) return zerr(ZE_GENERIC);
  return r;
}

static int compress_batch_device(zstdb200_ctx* ctx, int device_index, int level, int checksum, const void* src_base,
                                 const uint64_t* src_off, const uint32_t* src_size, void* dst_base, const uint64_t* dst_off,
                                 const uint32_t* dst_cap, uint32_t* result, size_t n, void* stream, bool useDict) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (device_index < 0 || device_index >= (int)ctx->dev.size()) { ctx->err = "bad device_index"; return 1; }
  if (level < 1 || level > 3) { ctx->err = "level must be 1..3"; return 1; }
  if (n > ctx->maxItems) { ctx->err = "n exceeds zstdb200_max_items"; return 1; }
  if (useDict && ctx->encDict.empty()) { ctx->err = "no dictionary loaded (zstdb200_load_dictionary)"; return 1; }
  Device& d = ctx->dev[device_index];
  CK(cudaSetDevice(d.id));
  u32 maxSrc = 0;
  if (device_max_u32(ctx, d, src_size, n, stream ? (cudaStream_t)stream : d.stream[0], &maxSrc)) return 1;
  EncodeArgs a{(const u8*)src_base, src_off, src_size, (u8*)dst_base, dst_off, dst_cap, result, (u32)n, 0, level, checksum, maxSrc, ENC_EXCLUSIVE};
  if (useDict) set_dict(ctx, d, a);
  int nl = 0;
  CK(encode_launch(a, d.enc, stream ? (cudaStream_t)stream : d.stream[0], &nl));
  ctx->launches += nl;
  return 0;
}

int zstdb200_compress_batch(zstdb200_ctx* ctx, int level, int checksum, const void* const* src, const uint32_t* srcSize,
                            void* const* dst, const uint32_t* dstCap, uint32_t* result, size_t n) {
  return compress_batch(ctx, level, checksum, src, srcSize, dst, dstCap, result, n, false);
}
int zstdb200_compress_batch_using_dict(zstdb200_ctx* ctx, int level, int checksum, const void* const* src, const uint32_t* srcSize,
                                       void* const* dst, const uint32_t* dstCap, uint32_t* result, size_t n) {
  return compress_batch(ctx, level, checksum, src, srcSize, dst, dstCap, result, n, true);
}
uint32_t zstdb200_compress(zstdb200_ctx* ctx, int level, int checksum, void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize) {
  return compress_one(ctx, level, checksum, dst, dstCapacity, src, srcSize, false);
}
uint32_t zstdb200_compress_using_dict(zstdb200_ctx* ctx, int level, int checksum, void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize) {
  return compress_one(ctx, level, checksum, dst, dstCapacity, src, srcSize, true);
}
int zstdb200_compress_batch_device(zstdb200_ctx* ctx, int device_index, int level, int checksum, const void* src_base,
                                   const uint64_t* src_off, const uint32_t* src_size, void* dst_base, const uint64_t* dst_off,
                                   const uint32_t* dst_cap, uint32_t* result, size_t n, void* stream) {
  return compress_batch_device(ctx, device_index, level, checksum, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream, false);
}
int zstdb200_compress_batch_device_using_dict(zstdb200_ctx* ctx, int device_index, int level, int checksum, const void* src_base,
                                              const uint64_t* src_off, const uint32_t* src_size, void* dst_base, const uint64_t* dst_off,
                                              const uint32_t* dst_cap, uint32_t* result, size_t n, void* stream) {
  return compress_batch_device(ctx, device_index, level, checksum, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream, true);
}

// zstdb200_compress_batch_device with CUDA events between its kernels (see zstdb200_decompress_batch_device_timed).
int zstdb200_compress_batch_device_timed(zstdb200_ctx* ctx, int device_index, int level, int checksum, const void* src_base,
                                         const uint64_t* src_off, const uint32_t* src_size, void* dst_base, const uint64_t* dst_off,
                                         const uint32_t* dst_cap, uint32_t* result, size_t n, void* stream, float* kernel_ms, int max_kernels) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (device_index < 0 || device_index >= (int)ctx->dev.size()) { ctx->err = "bad device_index"; return 1; }
  if (level < 1 || level > 3) { ctx->err = "level must be 1..3"; return 1; }
  if (n > ctx->maxItems) { ctx->err = "n exceeds zstdb200_max_items"; return 1; }
  Device& d = ctx->dev[device_index];
  CK(cudaSetDevice(d.id));
  cudaStream_t st = stream ? (cudaStream_t)stream : d.stream[0];
  EventSet<ENCODE_KERNELS + 1> es; CK(es.create());
  cudaEvent_t* ev = es.ev;
  u32 maxSrc = 0;
  if (device_max_u32(ctx, d, src_size, n, st, &maxSrc)) return 1;
  EncodeArgs a{(const u8*)src_base, src_off, src_size, (u8*)dst_base, dst_off, dst_cap, result, (u32)n, 0, level, checksum, maxSrc, ENC_EXCLUSIVE};
  int nl = 0;
  CK(encode_launch(a, d.enc, st, &nl, ev));
  ctx->launches += nl;
  CK(cudaStreamSynchronize(st));
  for (int k = 0; k < ENCODE_KERNELS && k < max_kernels; k++) CK(cudaEventElapsedTime(&kernel_ms[k], ev[k], ev[k + 1]));
  return 0;
}
const char* zstdb200_encode_kernel_name(int k) { return (k >= 0 && k < ENCODE_KERNELS) ? kEncodeKernelNames[k] : ""; }

uint32_t zstdb200_train_dictionary(zstdb200_ctx* ctx, void* dictBuffer, uint32_t dictCapacity, const void* samples,
                                   const uint32_t* sampleSizes, size_t nbSamples, zstdb200_train_params* params) {
  if (!ctx) return zerr(ZE_GENERIC);
  ctx->err.clear();
  if (!dictBuffer || (nbSamples && !sampleSizes)) { ctx->err = "null argument"; return zerr(ZE_GENERIC); }
  if (nbSamples > 0xFFFFFFFFull) { ctx->err = "too many samples"; return zerr(ZE_GENERIC); }
  zstdb200_train_params p{};
  if (params) p = *params;
  Device& d = ctx->dev[0];
  if (cudaSetDevice(d.id) != cudaSuccess) { ctx->err = "cudaSetDevice failed"; return zerr(ZE_GENERIC); }
  DtDevice dv{d.stream[0], &d.enc, d.d_dst, ctx->srcCap, d.d_result, d.h_result, d.d_desc, d.h_desc, ctx->maxBatch, ctx->maxItems, 0};
  const u32 r = dt_train_run(dv, (u8*)dictBuffer, dictCapacity, (const u8*)samples, sampleSizes, nbSamples, p, ctx->err);
  ctx->launches += dv.launches;
  if (!is_err(r) && params) { params->k = p.k; params->d = p.d; }
  return r;
}

void* zstdb200_host_alloc(size_t bytes) { void* p = nullptr; return cudaMallocHost(&p, bytes ? bytes : 1) == cudaSuccess ? p : nullptr; }
void zstdb200_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
