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
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/zstdb200.h"
#include "decode_kernels.cuh"
#include "dict_train.cuh"
#include "encode_kernels.cuh"
#include "host_plan.h"
#include "seekable.h"
#include "seekable_kernels.cuh"
#include "zb_encode.cuh"

using namespace zb;

namespace {

constexpr int NSTREAMS = 8;
static_assert(NSTREAMS <= ENC_STREAM_PARTS, "one encoder slot partition per stream");

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
  // Work that zstdb200_decompress_seekable_device left queued (it returns without synchronising) still reads the pinned
  // h_desc / h_seek and the device's descriptors, arenas and scratch: every later call that writes them, from the CPU or on
  // another stream, first waits for pendingEv (pending_wait).
  cudaEvent_t pendingEv = nullptr; bool pending = false;
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
  u8* d_seek = nullptr; u8* h_seek = nullptr;   // seekable archives (seek_scratch), allocated by their first call
  // pinned host memory
  u8 *h_src = nullptr, *h_dst = nullptr;
  u8* h_desc = nullptr;
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
  // waits for the last event, then ms[k] = time from event k to event k + 1 (at most max of them)
  cudaError_t read(float* ms, int max) {
    cudaError_t e = cudaEventSynchronize(ev[N - 1]);
    for (int k = 0; e == cudaSuccess && k < N - 1 && k < max; k++) e = cudaEventElapsedTime(&ms[k], ev[k], ev[k + 1]);
    return e;
  }
};

// CUDA errors of the entry points (ctx->err, return 1) and of the steps of a sub-batch (returned as text)
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { char b_[512]; snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", \
                      #call, cudaGetErrorString(e_), __FILE__, __LINE__); ctx->err = b_; return 1; } } while (0)
#define SB_CK(call, what) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return std::string(what) + ": " + cudaGetErrorString(e_); } while (0)
#define SB_TRY(step) do { std::string r_ = (step); if (!r_.empty()) return r_; } while (0)

int alloc_device(zstdb200_ctx* ctx, Device& d) {
  CK(cudaSetDevice(d.id));
  for (auto& s : d.stream) CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&d.descEv, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&d.pendingEv, cudaEventDisableTiming));
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
  cudaFree(d.d_seek); cudaFreeHost(d.h_seek);
  encode_free(d.enc);
  cudaFreeHost(d.h_src); cudaFreeHost(d.h_dst); cudaFreeHost(d.h_desc);
  for (auto& s : d.stream) if (s) cudaStreamDestroy(s);
  if (d.descEv) cudaEventDestroy(d.descEv);
  if (d.pendingEv) cudaEventDestroy(d.pendingEv);
  for (auto& ev : d.sliceEv) cudaEventDestroy(ev);
}

// Waits until no work a call left queued uses the device's staging and scratch (Device::pendingEv).
cudaError_t pending_wait(Device& d) {
  if (!d.pending) return cudaSuccess;
  d.pending = false;
  return cudaEventSynchronize(d.pendingEv);
}

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

enum class Op { Decompress, Compress };

// Items that hold several data frames (DecompressMultiFrame, ZStdDecompress.cs:2096-2160): each pass from a.pass on decodes
// the next data frame of every item and counts in *a.more (slot `slot`) the items with another; passes run until none has.
// `st` is synchronised once per pass (the count has to reach the host).  marks: as for decode_launch, first pass only.
cudaError_t decode_passes(Device& d, DecodeArgs a, u32 slot, cudaStream_t st, int* launches, cudaEvent_t* marks = nullptr) {
  cudaError_t e;
  for (;; a.pass++, marks = nullptr) {
    if ((e = cudaMemsetAsync(a.more, 0, 4, st)) != cudaSuccess) return e;
    if ((e = decode_launch(a, st, launches, marks)) != cudaSuccess) return e;
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
  struct SeekJob* seek = nullptr;   // seekable archives (below); null for every other call
};

// Seekable archives (seekable.h) through the host batch path.
struct SeekJob {
  // compress: after its encode, each sub-batch packs its frames on the device (k_seek_pack).  Once its result codes are on the
  // host it waits until the sub-batch before it has published where it ends (start[lo], lo: its first item), publishes its own
  // end (start[lo + m]) and copies its span to out + start[lo]: every byte crosses PCIe once and lands in its final place, also
  // when devices run concurrently.  ~0: not known yet.  A device that fails calls abort(), which releases every waiter.
  u8* out = nullptr;
  std::vector<u64> start;
  std::mutex mu; std::condition_variable cv; bool aborted = false;
  bool wait_start(size_t lo, u64* at) {
    std::unique_lock<std::mutex> l(mu);
    cv.wait(l, [&] { return aborted || start[lo] != ~0ull; });
    *at = start[lo];
    return !aborted;
  }
  void publish(size_t i, u64 v) { { std::lock_guard<std::mutex> l(mu); start[i] = v; } cv.notify_all(); }
  void abort() { { std::lock_guard<std::mutex> l(mu); aborted = true; } cv.notify_all(); }
  // decompress: each slice's frames are checked against their table entries right after their decode, while the bytes are on
  // the device (k_seek_check); cksum[i] is the entry's checksum of item i, null when the table carries none
  const u32* cksum = nullptr;
};

// The seekable calls' per-device scratch: d_seek = [offsets (maxItems + 2) x 8][cksum maxItems x 4][frame maxItems x 4]
// [first 8][done 4]; h_seek (pinned) = [cksum maxItems x 4][frame maxItems x 4][footer 16]
struct SeekScratch {
  u64* offsets; u32* cksum; u32* frame; unsigned long long* first; u32* done;
  u32* h_cksum; u32* h_frame; u8* h_footer;
};
size_t seek_device_bytes(size_t items) { return (items + 2) * 8 + items * 8 + 16; }
SeekScratch seek_scratch(const zstdb200_ctx* ctx, const Device& d) {
  const size_t items = ctx->maxItems;
  SeekScratch s;
  s.offsets = (u64*)d.d_seek; s.cksum = (u32*)(s.offsets + items + 2); s.frame = s.cksum + items;
  s.first = (unsigned long long*)(s.frame + items); s.done = (u32*)(s.first + 1);
  s.h_cksum = (u32*)d.h_seek; s.h_frame = s.h_cksum + items; s.h_footer = (u8*)(s.h_frame + items);
  return s;
}
int seek_alloc(zstdb200_ctx* ctx, Device& d) {
  if (d.d_seek) return 0;
  CK(cudaSetDevice(d.id));
  CK(cudaMalloc(&d.d_seek, seek_device_bytes(ctx->maxItems)));
  CK(cudaMallocHost(&d.h_seek, ctx->maxItems * 8 + 16));
  return 0;
}

// The arguments of one decode launch over n items, numbered from item_base in the arenas, on stream slot `slot` (its counters
// and Huffman full-table region).  The item lists are indexed by item_base, so slices of one sub-batch that run concurrently
// use disjoint ranges of them.  ZSTDB200_PAR=0 keeps every frame on the frame-serial kernels (A/B measurements).
DecodeArgs decode_args(const zstdb200_ctx* ctx, const Device& d, const Items& it, size_t n, u32 item_base, u32 slot) {
  static const bool par = env_int("ZSTDB200_PAR", 1, 0, 1) != 0;
  static const u32 seqAMax = (u32)env_int("ZSTDB200_SEQ_A_MAX", 512, 0, 0x7FFFFFFF), seqBMax = (u32)env_int("ZSTDB200_SEQ_B_MAX", 2048, 0, 0x7FFFFFFF);
  DecodeArgs a{};
  a.src_base = it.src; a.src_off = it.srcOff; a.src_size = it.srcSize;
  a.dst_base = it.dst; a.dst_off = it.dstOff; a.dst_cap = it.dstCap; a.result = it.result;
  a.n = (u32)n; a.item_base = item_base; a.info = d.d_info + item_base; a.lit_arena = d.d_lit; a.seq_arena = d.d_seq;
  a.dict = d.dictOn ? d.d_dictState : nullptr; a.dict_bytes = d.d_dict; a.pass = 0; a.more = d.d_more + slot;
  a.units = par ? d.d_units : nullptr; a.par_list = d.d_parList; a.list_stride = (u32)(ctx->maxItems + 1); a.cnt = d.d_cnt + 8 * slot;
  a.seq_a_max = seqAMax; a.seq_b_max = seqBMax; a.huf_full = (u16*)(d.d_hufFull + d.hufFullBytes * slot);
  return a;
}

// One sub-batch [lo, hi) on one device and its plan (host_plan.h): direct DMA where the caller's layout allows, the
// descriptors, the slices.  The steps return "" or an error description.
struct SubBatch {
  zstdb200_ctx* ctx; Device& d; const Job& j;
  size_t lo, m; bool decode, srcDirect, dstDirect, eager;
  bool packed;                   // a seekable compress: no per-item output; the frames leave packed, once (pack / fetch_packed)
  const u8* srcBase; u8* dstBase;
  DescView h;                    // the descriptors (device offsets) in the pinned staging
  Items dev;                     // the items on the device
  std::vector<Range> slices;

  SubBatch(zstdb200_ctx* c, Device& dv, const Job& jb, size_t lo_, size_t hi)
      : ctx(c), d(dv), j(jb), lo(lo_), m(hi - lo_), decode(jb.op == Op::Decompress), packed(jb.seek && !decode),
        srcBase((const u8*)jb.src[lo_]), dstBase((u8*)jb.dst[lo_]), h(dv.h_desc, hi - lo_) {
    // pageable caller memory goes through the pinned staging with parallel host copies (a pageable cudaMemcpyAsync
    // is a synchronous, single-threaded bounce inside the driver)
    const size_t inLim = decode ? ctx->srcCap : ctx->dstSpan, outLim = decode ? ctx->dstSpan : ctx->srcCap;
    srcDirect = back_to_back(j.src + lo, j.srcSize + lo, m, 64, inLim) && is_dma_able(srcBase);
    dstDirect = std::equal(j.effCap + lo, j.effCap + hi, j.dstCap + lo) && back_to_back(j.dst + lo, j.dstCap + lo, m, 0, outLim) &&
                is_dma_able(dstBase);
    size_t in = 0, out = 0;
    for (size_t k = 0; k < m; k++) {
      const size_t i = lo + k;
      h.srcSize[k] = j.srcSize[i]; h.dstCap[k] = j.effCap[i];
      h.srcOff[k] = srcDirect ? (u64)((const u8*)j.src[i] - srcBase) : in;
      h.dstOff[k] = dstDirect ? (u64)((u8*)j.dst[i] - dstBase) : out;
      in += align_up(j.srcSize[i], 16); out += align_up(j.effCap[i], 16);
    }
    dev = DescView(d.d_desc, m).items(d.d_src, d.d_dst, d.d_result);
    static const size_t sliceBytes = (size_t)env_int("ZSTDB200_SLICE_MB", (int)(SLICE_BYTES_DEFAULT >> 20), 1, 4096) << 20;
    slices = plan_slices(h.srcSize, h.dstCap, m, decode, sliceBytes);
    eager = !dstDirect && decode && slices.size() > 1;
  }

  // Small copies cost the copy engines about as much as a megabyte each, and they queue between the slices'
  // payload copies: descriptors go up once per sub-batch, results and counters come back once at its end.
  std::string start() {
    cudaStream_t s0 = d.stream[0];
    SB_CK(cudaMemsetAsync(d.d_more, 0, NSTREAMS * 4, s0), "memset");
    SB_CK(cudaMemcpyAsync(d.d_desc, d.h_desc, DescView::bytes(m), cudaMemcpyHostToDevice, s0), "H2D desc");
    if (decode && j.seek && j.seek->cksum) {   // the table's checksums of the sub-batch's frames, for k_seek_check
      const SeekScratch sc = seek_scratch(ctx, d);
      memcpy(sc.h_cksum, j.seek->cksum + lo, m * 4);
      SB_CK(cudaMemcpyAsync(sc.cksum, sc.h_cksum, m * 4, cudaMemcpyHostToDevice, s0), "H2D checksums");
    }
    if (slices.size() > 1) {
      SB_CK(cudaEventRecord(d.descEv, s0), "event");
      for (int k = 1; k < NSTREAMS; k++) SB_CK(cudaStreamWaitEvent(d.stream[k], d.descEv, 0), "event wait");
    }
    if (eager) while (d.sliceEv.size() < slices.size()) { cudaEvent_t ev; SB_CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming), "event create"); d.sliceEv.push_back(ev); }
    return "";
  }

  std::string stage_in(size_t a, size_t b, cudaStream_t st) {
    const size_t inLo = h.srcOff[a], inHi = h.srcOff[b - 1] + h.srcSize[b - 1];
    if (!srcDirect) parallel_for(b - a, inHi - inLo, [&](size_t x, size_t y) {
      for (size_t k = a + x; k < a + y; k++) if (h.srcSize[k]) memcpy(d.h_src + h.srcOff[k], j.src[lo + k], h.srcSize[k]);
    });
    if (inHi > inLo) SB_CK(cudaMemcpyAsync(d.d_src + inLo, (srcDirect ? srcBase : d.h_src) + inLo, inHi - inLo, cudaMemcpyHostToDevice, st), "H2D src");
    return "";
  }

  std::string launch(size_t a, size_t b, u32 slot, cudaStream_t st, uint64_t* launches) {
    int nl = 0;
    cudaError_t e;
    if (decode) {
      DecodeArgs da = decode_args(ctx, d, dev.from(a), b - a, (u32)a, slot);
      if (j.seek) da.more = nullptr;   // a seek table entry is one frame: nothing behind it is decoded
      e = decode_launch(da, st, &nl);
      if (e == cudaSuccess && j.seek) {
        const SeekScratch sc = seek_scratch(ctx, d);
        e = seek_check({dev.from(a), da.info, (u32)(b - a), j.seek->cksum ? sc.cksum + a : nullptr, nullptr, nullptr, nullptr, 0, nullptr, 0},
                       st, &nl);
      }
    } else {
      e = encode_launch(encode_args(dev.from(a), b - a, (u32)a, j.level, j.checksum, j.maxSrc, slot, j.useDict ? d.d_encDict : nullptr,
                                    &ctx->encDict), d.enc, st, &nl);
    }
    *launches += nl;
    SB_CK(e, "kernel launch");
    return "";
  }

  // Seekable compress: the sub-batch's frames, back to back from d_src[0] (the raw chunks there are no longer needed)
  std::string pack(uint64_t* launches) {
    int nl = 0;
    const SeekScratch sc = seek_scratch(ctx, d);
    const cudaError_t e = seek_pack({d.d_dst, dev.dstOff, dev.result, dev.srcSize, (u32)m, d.d_src, sc.offsets, nullptr, 0, j.checksum},
                                    d.stream[0], &nl);
    *launches += nl;
    SB_CK(e, "pack launch");
    return "";
  }

  // ... and their one copy to the host, at their final offset (SeekJob).  A failed frame packs nothing; the call then fails.
  std::string fetch_packed() {
    u64 total = 0, at;
    bool failed = false;
    for (size_t k = 0; k < m; k++) { failed |= is_err(d.h_result[k]); total += d.h_result[k]; }
    if (!j.seek->wait_start(lo, &at)) return "";   // an earlier sub-batch's device failed: so does the call
    j.seek->publish(lo + m, failed ? at : at + total);
    if (failed) return "";
    u8* to = j.seek->out + at;
    const bool direct = is_dma_able(to);
    if (total) SB_CK(cudaMemcpyAsync(direct ? to : d.h_dst, d.d_src, total, cudaMemcpyDeviceToHost, d.stream[0]), "D2H packed");
    SB_CK(cudaStreamSynchronize(d.stream[0]), "stream sync");
    if (!direct) parallel_for((total + (1u << 20) - 1) >> 20, total, [&](size_t x, size_t y) {
      const size_t a = x << 20, b = std::min<size_t>(total, y << 20);
      if (b > a) memcpy(to + a, d.h_dst + a, b - a);
    });
    return "";
  }

  std::string stage_out(size_t a, size_t b, cudaStream_t st) {
    const size_t outLo = h.dstOff[a], outHi = h.dstOff[b - 1] + h.dstCap[b - 1];
    if (outHi > outLo) SB_CK(cudaMemcpyAsync((dstDirect ? dstBase : d.h_dst) + outLo, d.d_dst + outLo, outHi - outLo, cudaMemcpyDeviceToHost, st), "D2H dst");
    return "";
  }

  std::string finish(uint64_t* launches) {
    // Pageable destinations of a decode: scatter every slice out of the pinned staging as soon as its copy has landed,
    // while the later slices are still in flight (the whole capacity of each item is copied: the result codes only arrive
    // at the end; bytes past result[i] are unspecified, include/zstdb200.h).
    for (size_t s = 0; eager && s < slices.size(); s++) {
      SB_CK(cudaEventSynchronize(d.sliceEv[s]), "event sync");
      const size_t a = slices[s].lo, b = slices[s].hi;
      parallel_for(b - a, h.dstOff[b - 1] + h.dstCap[b - 1] - h.dstOff[a], [&](size_t x, size_t y) {
        for (size_t k = a + x; k < a + y; k++) if (h.dstCap[k]) memcpy(j.dst[lo + k], d.h_dst + h.dstOff[k], h.dstCap[k]);
      });
    }
    // a single slice ran on stream 0 alone: its results ride the same stream and one synchronisation ends the call
    if (slices.size() > 1) for (auto& st : d.stream) SB_CK(cudaStreamSynchronize(st), "stream sync");
    if (packed) SB_TRY(pack(launches));
    SB_CK(cudaMemcpyAsync(d.h_more, d.d_more, (NSTREAMS + m) * 4, cudaMemcpyDeviceToHost, d.stream[0]), "D2H results");
    SB_CK(cudaStreamSynchronize(d.stream[0]), "stream sync");
    u32 anyMore = 0;
    for (int k = 0; k < NSTREAMS; k++) anyMore |= d.h_more[k];
    if (decode && anyMore) {
      // rare path: some items hold several data frames.  Everything is still resident: decode the remaining frames
      // pass by pass over the whole sub-batch, then fetch results and output again.
      cudaStream_t st = d.stream[0]; int nl = 0;
      DecodeArgs a = decode_args(ctx, d, dev, m, 0, 0); a.pass = 1;
      const cudaError_t e = decode_passes(d, a, 0, st, &nl);
      *launches += nl;
      SB_CK(e, "multi-frame passes");
      SB_CK(cudaMemcpyAsync(d.h_result, d.d_result, m * 4, cudaMemcpyDeviceToHost, st), "D2H result");
      SB_TRY(stage_out(0, m, st));
      SB_CK(cudaStreamSynchronize(st), "stream sync");
    }
    for (size_t k = 0; k < m; k++) j.result[lo + k] = d.h_result[k];
    if (packed) return fetch_packed();
    // staged output not scattered yet (compress: frames are much smaller than their capacity; single-slice calls; items
    // that needed further passes): copy what was produced; on error the reference leaves dst partially written, we copy nothing
    if (!dstDirect && (!eager || anyMore)) parallel_for(m, h.dstOff[m - 1] + h.dstCap[m - 1], [&](size_t x, size_t y) {
      for (size_t k = x; k < y; k++) {
        const size_t i = lo + k; const u32 r = d.h_result[k];
        if (!is_err(r) && r) memcpy(j.dst[i], d.h_dst + h.dstOff[k], std::min<u32>(r, j.dstCap[i]));
      }
    });
    return "";
  }
};

// Descriptors up in one copy, then stage in / launch / stage out per slice, the slices dealt round-robin to the streams, then
// finish.
std::string run_subbatch(zstdb200_ctx* ctx, Device& d, const Job& j, size_t lo, size_t hi, uint64_t* launches) {
  static const int nStreams = env_int("ZSTDB200_STREAMS", NSTREAMS, 1, NSTREAMS);
  SB_CK(pending_wait(d), "pending wait");
  SubBatch sb(ctx, d, j, lo, hi);
  SB_TRY(sb.start());
  for (size_t s = 0; s < sb.slices.size(); s++) {
    const size_t a = sb.slices[s].lo, b = sb.slices[s].hi;
    const u32 slot = (u32)(s % nStreams);
    cudaStream_t st = d.stream[slot];
    SB_TRY(sb.stage_in(a, b, st));
    SB_TRY(sb.launch(a, b, slot, st, launches));
    if (!sb.packed) SB_TRY(sb.stage_out(a, b, st));
    if (sb.eager) SB_CK(cudaEventRecord(d.sliceEv[s], st), "event");
  }
  return sb.finish(launches);
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
  subs = split_over_devices(std::move(subs), nd, [&](size_t i) { return (uint64_t)j.srcSize[i] + j.effCap[i] + 1; });
  std::vector<std::string> errs(nd);
  std::vector<uint64_t> launches(nd, 0);
  auto worker = [&](size_t di) {
    Device& d = ctx->dev[di];
    cudaError_t e = cudaSetDevice(d.id);
    if (e != cudaSuccess) errs[di] = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
    for (size_t s = di; errs[di].empty() && s < subs.size(); s += nd) errs[di] = run_subbatch(ctx, d, j, subs[s].lo, subs[s].hi, &launches[di]);
    if (!errs[di].empty() && j.seek) j.seek->abort();   // other devices' sub-batches may wait for this one's place (SeekJob)
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

// Compression levels: 1..3, and -7..-1 (libzstd's fast negative levels, acceleration = -level)
static bool level_ok(int level) { return (level >= 1 && level <= 3) || (level >= -7 && level <= -1); }
static const char* const kLevelError = "level must be 1..3 or -7..-1";

// The checks every device-pointer entry point starts with (compress: the level and a loaded dictionary too); then the device
// is selected.  *st: the caller's stream, or the device's first one.
int device_call(zstdb200_ctx* ctx, Op op, int device_index, size_t n, int level, bool useDict, void* stream, Device** d, cudaStream_t* st) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (device_index < 0 || device_index >= (int)ctx->dev.size()) { ctx->err = "bad device_index"; return 1; }
  if (op == Op::Compress && !level_ok(level)) { ctx->err = kLevelError; return 1; }
  if (n > ctx->maxItems) { ctx->err = "n exceeds zstdb200_max_items"; return 1; }
  if (useDict && ctx->encDict.empty()) { ctx->err = "no dictionary loaded (zstdb200_load_dictionary)"; return 1; }
  *d = &ctx->dev[device_index];
  CK(cudaSetDevice((*d)->id));
  CK(pending_wait(**d));
  *st = stream ? (cudaStream_t)stream : (*d)->stream[0];
  return 0;
}

// One item through a batch call.  A null array is an empty one (the C# shim passes null for byte[0]).
template <class F>
uint32_t one_item(void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize, F batch) {
  static unsigned char dummy[16];
  if (!src) { src = dummy; srcSize = 0; }
  if (!dst) { dst = dummy; dstCapacity = 0; }
  uint32_t r = zerr(ZE_GENERIC);
  return batch(&src, &srcSize, &dst, &dstCapacity, &r) ? zerr(ZE_GENERIC) : r;
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
    DictState ds{};
    dict_load_host((const u8*)dict, dictSize, ds);
    ctx->encDict = enc_dict_block((const u8*)dict, dictSize, ds);
  }
  for (auto& d : ctx->dev) {
    CK(cudaSetDevice(d.id));
    CK(pending_wait(d));
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
  return one_item(dst, dstCapacity, src, srcSize, [&](auto s, auto ss, auto d, auto dc, auto r) { return zstdb200_decompress_batch(ctx, s, ss, d, dc, r, 1); });
}

// Device-resident decode: one launch sequence over the whole batch on the caller's stream (slicing a resident batch
// over several streams was measured slower: whole-batch kernels fill the GPU better).  The count of items that
// hold a further data frame has to reach the host, so this entry point synchronises the stream once per pass.
static int decompress_device(zstdb200_ctx* ctx, int device_index, const void* src_base, const uint64_t* src_off, const uint32_t* src_size,
                             void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap, uint32_t* result, size_t n, void* stream,
                             EventSet<DECODE_KERNELS + 1>* es) {
  Device* d; cudaStream_t st;
  if (device_call(ctx, Op::Decompress, device_index, n, 0, false, stream, &d, &st)) return 1;
  if (es) CK(es->create());
  const DecodeArgs a = decode_args(ctx, *d, Items{(const u8*)src_base, src_off, src_size, (u8*)dst_base, dst_off, dst_cap, result}, n, 0, 0);
  int nl = 0;
  CK(decode_passes(*d, a, 0, st, &nl, es ? es->ev : nullptr));
  ctx->launches += nl;
  return 0;
}

int zstdb200_decompress_batch_device(zstdb200_ctx* ctx, int device_index, const void* src_base, const uint64_t* src_off,
                                     const uint32_t* src_size, void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                     uint32_t* result, size_t n, void* stream) {
  return decompress_device(ctx, device_index, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream, nullptr);
}

// Same work as one launch sequence with CUDA events between the kernels: per-kernel device times for the
// bench's roofline block.
int zstdb200_decompress_batch_device_timed(zstdb200_ctx* ctx, int device_index, const void* src_base, const uint64_t* src_off,
                                           const uint32_t* src_size, void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                           uint32_t* result, size_t n, void* stream, float* kernel_ms, int max_kernels) {
  EventSet<DECODE_KERNELS + 1> es;
  if (decompress_device(ctx, device_index, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream, &es)) return 1;
  CK(es.read(kernel_ms, max_kernels));
  return 0;
}
const char* zstdb200_decode_kernel_name(int k) { return (k >= 0 && k < DECODE_KERNELS) ? kDecodeKernelNames[k] : ""; }

size_t zstdb200_compress_bound(size_t srcSize) { return encode_bound(srcSize); }

// The compress entry points with and without the context's dictionary share these bodies (useDict).
static int compress_batch(zstdb200_ctx* ctx, int level, int checksum, const void* const* src, const uint32_t* srcSize,
                          void* const* dst, const uint32_t* dstCap, uint32_t* result, size_t n, bool useDict) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (!level_ok(level)) { ctx->err = kLevelError; return 1; }
  if (useDict && ctx->encDict.empty()) { ctx->err = "no dictionary loaded (zstdb200_load_dictionary)"; return 1; }
  Job j{Op::Compress, level, checksum, src, srcSize, dst, dstCap, result, nullptr, 0, useDict};
  return run_host_batch(ctx, j, n);
}

static int compress_device(zstdb200_ctx* ctx, int device_index, int level, int checksum, const void* src_base, const uint64_t* src_off,
                           const uint32_t* src_size, void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap, uint32_t* result,
                           size_t n, void* stream, bool useDict, EventSet<ENCODE_KERNELS + 1>* es) {
  Device* d; cudaStream_t st;
  if (device_call(ctx, Op::Compress, device_index, n, level, useDict, stream, &d, &st)) return 1;
  if (es) CK(es->create());
  // the largest chunk of the call selects the match stage's table sizes: the size array comes to the host once (one small
  // copy and one synchronisation of the stream)
  u32 maxSrc = 0;
  if (n) {
    CK(cudaMemcpyAsync(d->h_desc, src_size, n * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    maxSrc = *std::max_element((const u32*)d->h_desc, (const u32*)d->h_desc + n);
  }
  const Items it{(const u8*)src_base, src_off, src_size, (u8*)dst_base, dst_off, dst_cap, result};
  int nl = 0;
  CK(encode_launch(encode_args(it, n, 0, level, checksum, maxSrc, ENC_EXCLUSIVE, useDict ? d->d_encDict : nullptr, &ctx->encDict), d->enc,
                   st, &nl, es ? es->ev : nullptr));
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
  return one_item(dst, dstCapacity, src, srcSize, [&](auto s, auto ss, auto d, auto dc, auto r) { return compress_batch(ctx, level, checksum, s, ss, d, dc, r, 1, false); });
}
uint32_t zstdb200_compress_using_dict(zstdb200_ctx* ctx, int level, int checksum, void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize) {
  return one_item(dst, dstCapacity, src, srcSize, [&](auto s, auto ss, auto d, auto dc, auto r) { return compress_batch(ctx, level, checksum, s, ss, d, dc, r, 1, true); });
}
int zstdb200_compress_batch_device(zstdb200_ctx* ctx, int device_index, int level, int checksum, const void* src_base,
                                   const uint64_t* src_off, const uint32_t* src_size, void* dst_base, const uint64_t* dst_off,
                                   const uint32_t* dst_cap, uint32_t* result, size_t n, void* stream) {
  return compress_device(ctx, device_index, level, checksum, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream, false, nullptr);
}
int zstdb200_compress_batch_device_using_dict(zstdb200_ctx* ctx, int device_index, int level, int checksum, const void* src_base,
                                              const uint64_t* src_off, const uint32_t* src_size, void* dst_base, const uint64_t* dst_off,
                                              const uint32_t* dst_cap, uint32_t* result, size_t n, void* stream) {
  return compress_device(ctx, device_index, level, checksum, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream, true, nullptr);
}

// zstdb200_compress_batch_device with CUDA events between its kernels (see zstdb200_decompress_batch_device_timed).
int zstdb200_compress_batch_device_timed(zstdb200_ctx* ctx, int device_index, int level, int checksum, const void* src_base,
                                         const uint64_t* src_off, const uint32_t* src_size, void* dst_base, const uint64_t* dst_off,
                                         const uint32_t* dst_cap, uint32_t* result, size_t n, void* stream, float* kernel_ms, int max_kernels) {
  EventSet<ENCODE_KERNELS + 1> es;
  if (compress_device(ctx, device_index, level, checksum, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream, false, &es))
    return 1;
  CK(es.read(kernel_ms, max_kernels));
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
  if (pending_wait(d) != cudaSuccess) { ctx->err = "waiting for queued work failed"; return zerr(ZE_GENERIC); }
  DtDevice dv{d.stream[0], &d.enc, d.d_dst, ctx->srcCap, d.d_result, d.h_result, d.d_desc, d.h_desc, ctx->maxBatch, ctx->maxItems, 0};
  const u32 r = dt_train_run(dv, (u8*)dictBuffer, dictCapacity, (const u8*)samples, sampleSizes, nbSamples, p, ctx->err);
  ctx->launches += dv.launches;
  if (!is_err(r) && params) { params->k = p.k; params->d = p.d; }
  return r;
}

// ---- seekable archives (seekable.h, seekable_kernels.cu) ---------------------------------------------------------------

uint32_t zstdb200_seekable_info_get(const void* src, uint64_t srcSize, zstdb200_seekable_info* info) {
  seek::Table t;
  const u32 r = seek::parse((const u8*)src, srcSize, &t);
  if (r) return r;
  if (info) *info = {t.contentSize, t.dataSize, t.n, t.ck ? 1u : 0u, t.maxContent, t.maxCompressed};
  return 0;
}

uint64_t zstdb200_seekable_bound(uint64_t srcSize, uint32_t frameSize) {
  if (frameSize == 0) return 0;
  return seek::bound(srcSize, frameSize, [](uint64_t c) { return (uint64_t)encode_bound(c); });
}

}  // extern "C"

namespace {

// The argument checks both seekable compress calls share.
int seek_compress_args(zstdb200_ctx* ctx, int checksum, uint32_t frameSize, const void* src, uint64_t srcSize, const void* dst,
                       uint64_t dstCapacity, const void* dstSize) {
  if ((!src && srcSize) || !dst || !dstSize) { ctx->err = "null argument"; return 1; }
  if (frameSize == 0 || frameSize > ctx->maxBatch) { ctx->err = "frameSize must be 1..max_batch_bytes"; return 1; }
  if (!seek::table_fits(seek::frame_count(srcSize, frameSize), checksum != 0)) {
    ctx->err = "too many frames: the seek table's Frame_Size would not fit 32 bits"; return 1;
  }
  if (dstCapacity < zstdb200_seekable_bound(srcSize, frameSize)) { ctx->err = "dstCapacity is below zstdb200_seekable_bound"; return 1; }
  return 0;
}

// A selected frame whose content does not fit one launch's arenas fails the call.
int seek_frames_fit(zstdb200_ctx* ctx, const std::vector<seek::Piece>& pieces) {
  for (auto& p : pieces)
    if (p.dsize > ctx->maxBatch || p.csize > ctx->maxBatch) { ctx->err = "a frame is larger than the context's max_batch_bytes"; return 1; }
  return 0;
}

}  // namespace

extern "C" {

int zstdb200_compress_seekable(zstdb200_ctx* ctx, int level, int checksum, uint32_t frameSize, const void* src, uint64_t srcSize,
                               void* dst, uint64_t dstCapacity, uint64_t* dstSize) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (!level_ok(level)) { ctx->err = kLevelError; return 1; }
  if (seek_compress_args(ctx, checksum, frameSize, src, srcSize, dst, dstCapacity, dstSize)) return 1;
  const size_t n = (size_t)seek::frame_count(srcSize, frameSize);
  const u8* s = (const u8*)src; u8* out = (u8*)dst;
  std::vector<const void*> srcs(n); std::vector<void*> dsts(n, nullptr);
  std::vector<uint32_t> sizes(n), caps(n), res(n);
  for (size_t i = 0; i < n; i++) {
    srcs[i] = s + (u64)i * frameSize; sizes[i] = seek::frame_content(srcSize, frameSize, i);
    caps[i] = (uint32_t)encode_bound(sizes[i]);
  }
  SeekJob sj; sj.out = out; sj.start.assign(n + 1, ~0ull); sj.start[0] = 0;
  Job j{Op::Compress, level, checksum ? 1 : 0, srcs.data(), sizes.data(), dsts.data(), caps.data(), res.data(), nullptr, 0, false, &sj};
  if (n) {
    for (auto& d : ctx->dev) if (seek_alloc(ctx, d)) return 1;
    if (run_host_batch(ctx, j, n)) return 1;
  }
  for (size_t i = 0; i < n; i++)
    if (is_err(res[i])) { ctx->err = "frame " + std::to_string(i) + " failed to compress: error " + std::to_string(zerr(res[i])); return 1; }
  // the frames are in place (SeekJob); the table from their sizes and each frame's own checksum
  const u64 total = sj.start[n];
  std::vector<uint32_t> cks(checksum ? n : 0);
  for (size_t i = 0, pos = 0; i < n; pos += res[i], i++) if (checksum) cks[i] = seek::rd32(out + pos + res[i] - 4);
  seek::write_table(out + total, n, res.data(), sizes.data(), cks.data(), checksum != 0);
  *dstSize = total + seek::table_bytes(n, checksum != 0);
  return 0;
}

// The frames are encoded into the context's staging (d_dst, 16-byte aligned slots of their compress bound), then packed into
// dst with their table.  One synchronisation: the descriptors' upload (as compress_batch_device's size fetch).
int zstdb200_compress_seekable_device(zstdb200_ctx* ctx, int device_index, int level, int checksum, uint32_t frameSize, const void* src,
                                      uint64_t srcSize, void* dst, uint64_t dstCapacity, uint64_t* dstSize, void* stream) {
  Device* d; cudaStream_t st;
  if (!ctx) return 1;
  const uint64_t nf = frameSize ? seek::frame_count(srcSize, frameSize) : 0;
  if (device_call(ctx, Op::Compress, device_index, (size_t)std::min<uint64_t>(nf, ~(size_t)0), level, false, stream, &d, &st)) return 1;
  if (seek_compress_args(ctx, checksum, frameSize, src, srcSize, dst, dstCapacity, dstSize)) return 1;
  if (srcSize > ctx->maxBatch) { ctx->err = "srcSize exceeds max_batch_bytes"; return 1; }
  if (seek_alloc(ctx, *d)) return 1;
  const size_t n = (size_t)nf;
  DescView h(d->h_desc, n);
  u64 out = 0;
  for (size_t i = 0; i < n; i++) {
    h.srcOff[i] = (u64)i * frameSize; h.srcSize[i] = seek::frame_content(srcSize, frameSize, i);
    h.dstCap[i] = (u32)encode_bound(h.srcSize[i]); h.dstOff[i] = out; out += align_up(h.dstCap[i], 16);
  }
  if (out > ctx->srcCap) { ctx->err = "the frames' compress bounds exceed the context's staging"; return 1; }
  int nl = 0;
  const DescView dv(d->d_desc, n);
  if (n) {
    CK(cudaMemcpyAsync(d->d_desc, d->h_desc, DescView::bytes(n), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));   // h_desc is the context's: the copy must be done before the next call refills it
    const Items it = dv.items((const u8*)src, d->d_dst, d->d_result);
    CK(encode_launch(encode_args(it, n, 0, level, checksum ? 1 : 0, (u32)std::min<uint64_t>(frameSize, srcSize), ENC_EXCLUSIVE, nullptr,
                                 &ctx->encDict), d->enc, st, &nl));
  }
  const SeekScratch sc = seek_scratch(ctx, *d);
  CK(seek_pack({d->d_dst, dv.dstOff, d->d_result, dv.srcSize, (u32)n, (u8*)dst, sc.offsets, dstSize, 1, checksum ? 1 : 0}, st, &nl));
  ctx->launches += nl;
  return 0;
}

int zstdb200_decompress_seekable(zstdb200_ctx* ctx, void* dst, uint64_t offset, uint64_t length, const void* src, uint64_t srcSize,
                                 uint32_t* code) {
  if (!ctx) return 1;
  ctx->err.clear();
  if (!code || (!src && srcSize) || (!dst && length)) { ctx->err = "null argument"; return 1; }
  seek::Table t; std::vector<seek::Piece> pieces;
  u32 r = seek::parse((const u8*)src, srcSize, &t);
  if (!r) r = seek::plan_range(t, offset, length, &pieces);
  *code = r;
  if (r || pieces.empty()) return 0;
  if (seek_frames_fit(ctx, pieces)) return 1;
  for (auto& d : ctx->dev) if (seek_alloc(ctx, d)) return 1;
  // one item per frame: interior frames decode straight into dst, the edge frames into scratch
  const size_t n = pieces.size();
  std::vector<const void*> srcs(n); std::vector<void*> dsts(n); std::vector<uint32_t> sizes(n), caps(n), res(n), cks(n);
  std::vector<std::vector<u8>> edge(n);
  for (size_t k = 0; k < n; k++) {
    const seek::Piece& p = pieces[k];
    if (p.edge()) edge[k].resize(p.dsize);
    srcs[k] = (const u8*)src + p.srcOff; sizes[k] = p.csize; caps[k] = p.dsize;
    dsts[k] = p.edge() ? (void*)edge[k].data() : (void*)((u8*)dst + p.dstOff);
    cks[k] = t.ck ? t.cksum[p.frame] : 0;
  }
  SeekJob sj; sj.cksum = t.ck ? cks.data() : nullptr;
  Job j{Op::Decompress, 0, 0, srcs.data(), sizes.data(), dsts.data(), caps.data(), res.data(), nullptr, 0, false, &sj};
  if (run_host_batch(ctx, j, n, false)) return 1;   // capacities are the entries' sizes: nothing to clamp
  for (size_t k = 0; k < n; k++) if (is_err(res[k])) { *code = res[k]; return 0; }
  for (size_t k = 0; k < n; k++) if (pieces[k].edge()) memcpy((u8*)dst + pieces[k].dstOff, edge[k].data() + pieces[k].skip, pieces[k].take);
  return 0;
}

// Edge frames first, into the context's staging d_dst, then the others in archive order straight into dst; each group is one
// launch sequence of the decode pipeline followed by k_seek_check.  The groups respect one launch's arenas and share one
// descriptor upload while they fit max_items (otherwise the stream is synchronised before the pinned descriptors are refilled).
int zstdb200_decompress_seekable_device(zstdb200_ctx* ctx, int device_index, void* dst, uint64_t offset, uint64_t length, const void* src,
                                        uint64_t srcSize, uint32_t* code, void* stream) {
  Device* d; cudaStream_t st;
  if (device_call(ctx, Op::Decompress, device_index, 0, 0, false, stream, &d, &st)) return 1;
  if (!code || (!src && srcSize) || (!dst && length)) { ctx->err = "null argument"; return 1; }
  if (seek_alloc(ctx, *d)) return 1;
  const SeekScratch sc = seek_scratch(ctx, *d);
  const u8* s = (const u8*)src;
  seek::Table t; std::vector<seek::Piece> pieces;
  u32 r = srcSize < seek::MIN_ARCHIVE ? seek::ERR_srcSize_wrong : 0;
  if (!r) {   // the footer, then the table: two small copies, two synchronisations
    CK(cudaMemcpyAsync(sc.h_footer, s + srcSize - seek::FOOTER_BYTES, seek::FOOTER_BYTES, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    seek::Footer f;
    r = seek::parse_footer(sc.h_footer, srcSize, &f);
    if (!r) {
      std::vector<u8> tab(f.tableBytes);
      CK(cudaMemcpyAsync(tab.data(), s + srcSize - f.tableBytes, f.tableBytes, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      r = seek::parse_table(tab.data(), srcSize, f, &t);
    }
  }
  if (!r) r = seek::plan_range(t, offset, length, &pieces);
  if (seek_frames_fit(ctx, pieces)) return 1;
  std::vector<size_t> order;   // indices into pieces: edge frames, then the rest
  for (size_t k = 0; k < pieces.size(); k++) if (pieces[k].edge()) order.push_back(k);
  const size_t nEdge = order.size();
  for (size_t k = 0; k < pieces.size(); k++) if (!pieces[k].edge()) order.push_back(k);
  bool big = false;
  auto bytes = [&](size_t x) { return (size_t)pieces[order[x]].dsize; };
  std::vector<Range> groups = make_subbatches(nEdge, ~(size_t)0, std::min(ctx->srcCap, ctx->maxBatch), ctx->maxItems, bytes, bytes, &big);
  std::vector<Range> inner = make_subbatches(order.size() - nEdge, ~(size_t)0, ctx->maxBatch, ctx->maxItems,
                                             [&](size_t x) { return bytes(nEdge + x); }, [&](size_t x) { return bytes(nEdge + x); }, &big);
  for (auto& g : inner) groups.push_back({nEdge + g.lo, nEdge + g.hi});
  u32 blocks = 0;
  for (auto& g : groups) blocks += seek_check_blocks((u32)(g.hi - g.lo));
  CK(cudaMemsetAsync(sc.first, 0xFF, 8, st));
  CK(cudaMemsetAsync(sc.done, 0, 4, st));
  int nl = 0;
  if (groups.empty()) {   // an error of the table or the range, or an empty range: only the code
    CK(seek_check({Items{}, nullptr, 0, nullptr, nullptr, sc.first, sc.done, 1, code, r}, st, &nl));
    CK(cudaEventRecord(d->pendingEv, st)); d->pending = true;
    ctx->launches += nl;
    return 0;
  }
  for (size_t g = 0; g < groups.size();) {
    size_t g1 = g, m = 0;
    while (g1 < groups.size() && m + (groups[g1].hi - groups[g1].lo) <= ctx->maxItems) m += groups[g1].hi - groups[g1].lo, g1++;
    CK(pending_wait(*d));   // the previous groups' work still reads the pinned descriptors
    DescView h(d->h_desc, m);
    for (size_t x = g, k = 0; x < g1; x++) {
      const bool isEdge = groups[x].lo < nEdge;
      u64 edgeAt = 0;
      const u64 base = isEdge ? 0 : pieces[order[groups[x].lo]].dstOff;
      for (size_t y = groups[x].lo; y < groups[x].hi; y++, k++) {
        const seek::Piece& p = pieces[order[y]];
        h.srcOff[k] = p.srcOff; h.srcSize[k] = p.csize; h.dstCap[k] = p.dsize;
        h.dstOff[k] = isEdge ? edgeAt : p.dstOff - base;
        edgeAt += align_up(p.dsize, 16);
        sc.h_frame[k] = p.frame; sc.h_cksum[k] = t.ck ? t.cksum[p.frame] : 0;
      }
    }
    CK(cudaMemcpyAsync(d->d_desc, d->h_desc, DescView::bytes(m), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(sc.frame, sc.h_frame, m * 4, cudaMemcpyHostToDevice, st));
    if (t.ck) CK(cudaMemcpyAsync(sc.cksum, sc.h_cksum, m * 4, cudaMemcpyHostToDevice, st));
    const DescView dv(d->d_desc, m);
    for (size_t x = g, k0 = 0; x < g1; k0 += groups[x].hi - groups[x].lo, x++) {
      const bool isEdge = groups[x].lo < nEdge;
      const u32 n = (u32)(groups[x].hi - groups[x].lo);
      u8* base = isEdge ? d->d_dst : (u8*)dst + pieces[order[groups[x].lo]].dstOff;
      const Items it = dv.items(s, base, d->d_result).from(k0);
      DecodeArgs a = decode_args(ctx, *d, it, n, 0, 0);
      a.more = nullptr;   // a seek table entry is one frame
      CK(decode_launch(a, st, &nl));
      CK(seek_check({it, a.info, n, t.ck ? sc.cksum + k0 : nullptr, sc.frame + k0, sc.first, sc.done, blocks, code, 0}, st, &nl));
      for (size_t k = k0; isEdge && k < k0 + n; k++) {
        const seek::Piece& p = pieces[order[groups[x].lo + (k - k0)]];
        CK(cudaMemcpyAsync((u8*)dst + p.dstOff, d->d_dst + h.dstOff[k] + p.skip, p.take, cudaMemcpyDeviceToDevice, st));
      }
    }
    CK(cudaEventRecord(d->pendingEv, st)); d->pending = true;
    g = g1;
  }
  ctx->launches += nl;
  return 0;
}

void* zstdb200_host_alloc(size_t bytes) { void* p = nullptr; return cudaMallocHost(&p, bytes ? bytes : 1) == cudaSuccess ? p : nullptr; }
void zstdb200_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
