// host_plan.h — how the host path of api.cu cuts a batch: sub-batches that fit the device arenas, their share per device,
// slices per stream, the descriptor layout and which caller buffers can be copied directly.  Pure functions over sizes and
// addresses (no CUDA), so that tests/hostsim/host_plan.cpp can check them on a CPU.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <algorithm>
#include <vector>

namespace zb {

constexpr size_t SLICE_BYTES_DEFAULT = 32u << 20;   // uncompressed bytes per slice (several slices per stream per GiB)
constexpr size_t MIN_SLICE_ITEMS_DECODE = 1024;      // and at least this many frames (decode kernels: one frame-time per launch)
constexpr size_t MIN_SLICE_ITEMS_ENCODE = 512;       // the match kernel fills the GPU with 2-4 thousand frames: start early

struct Range { size_t lo, hi; };

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// The data of one launch (device pointers): item i reads src[srcOff[i] .. + srcSize[i]) and writes at most dstCap[i] bytes
// at dst[dstOff[i] ..] and its result code at result[i].
struct Items {
  const uint8_t* src; const uint64_t* srcOff; const uint32_t* srcSize;
  uint8_t* dst; const uint64_t* dstOff; const uint32_t* dstCap; uint32_t* result;
  Items from(size_t a) const { return {src, srcOff + a, srcSize + a, dst, dstOff + a, dstCap + a, result + a}; }   // items a, a + 1, ..
};

// The descriptors of m items, laid out so that they travel in one copy: [srcOff m x 8][dstOff m x 8][srcSize m x 4][dstCap m x 4]
struct DescView {
  uint64_t* srcOff; uint64_t* dstOff; uint32_t* srcSize; uint32_t* dstCap;
  DescView(void* base, size_t m)
      : srcOff((uint64_t*)base), dstOff(srcOff + m), srcSize((uint32_t*)(dstOff + m)), dstCap(srcSize + m) {}
  static size_t bytes(size_t m) { return m * 24; }
  Items items(const uint8_t* src, uint8_t* dst, uint32_t* result) const { return {src, srcOff, srcSize, dst, dstOff, dstCap, result}; }
};

// Greedy split of [0, n) into consecutive sub-batches that respect the per-device arena limits.  Empty with *tooBig set when a
// single item exceeds the arena.
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
    if (hi == lo) { *tooBig = true; return r; }
    r.push_back({lo, hi}); lo = hi;
  }
  return r;
}

// Fewer sub-batches than devices: each is re-cut into up to nd parts so that every device gets a share.  Equal shares of
// cost(i) (bytes in + out), not of items: a raw-block frame costs a copy, a text frame a full decode.
template <class FC>
std::vector<Range> split_over_devices(std::vector<Range> subs, size_t nd, FC cost) {
  if (nd <= 1 || subs.size() >= nd) return subs;
  std::vector<Range> cut;
  for (auto& r : subs) {
    const size_t parts = std::min(nd, r.hi - r.lo);
    uint64_t total = 0;
    for (size_t i = r.lo; i < r.hi; i++) total += cost(i);
    size_t lo = r.lo; uint64_t acc = 0;
    for (size_t p = 0; p < parts; p++) {
      size_t hi = lo;
      const uint64_t want = total * (p + 1) / parts;
      while (hi < r.hi && (acc < want || hi == lo) && (r.hi - hi) > (parts - 1 - p)) { acc += cost(hi); hi++; }
      if (p + 1 == parts) hi = r.hi;
      cut.push_back({lo, hi}); lo = hi;
    }
  }
  return cut;
}

// Slices of a sub-batch of m items (srcSize / dstCap: its descriptors), dealt round-robin to the streams.  A slice is >=
// sliceBytes and >= MIN_SLICE_ITEMS frames: the kernels take one frame-time however few frames they are given, so slices of
// a few large frames would serialise on that latency.  Decode: the first slices are smaller (a quarter for two, a half for
// two more), because output can only start to leave once a slice's kernels are done (one frame-time however small the
// slice), and the D2H engine then has to be fed without a gap while the big slices finish.
inline std::vector<Range> plan_slices(const uint32_t* srcSize, const uint32_t* dstCap, size_t m, bool decode, size_t sliceBytes) {
  const size_t minItems = decode ? MIN_SLICE_ITEMS_DECODE : MIN_SLICE_ITEMS_ENCODE;
  std::vector<Range> slices;
  size_t a = 0;
  while (a < m) {
    const size_t k = slices.size(), shrink = decode ? (k < 2 ? 4 : (k < 4 ? 2 : 1)) : 1;
    const size_t wantItems = std::max<size_t>(1, minItems / shrink), wantBytes = sliceBytes / shrink;
    size_t b = a, bytes = 0;
    while (b < m && (b - a < wantItems || bytes + std::max(dstCap[b], srcSize[b]) <= wantBytes)) { bytes += std::max(dstCap[b], srcSize[b]); b++; }
    slices.push_back({a, b}); a = b;
  }
  return slices;
}

// True when the m buffers p[k] (size[k] bytes each) lie back to back in one span of at most `limit` bytes: each starts where
// the one before ends or at most `slack` bytes later.  Such buffers move with one copy per slice, without staging.
inline bool back_to_back(const void* const* p, const uint32_t* size, size_t m, size_t slack, size_t limit) {
  if (!p[0]) return false;
  for (size_t k = 0; k + 1 < m; k++) {
    const uint8_t *end = (const uint8_t*)p[k] + size[k], *next = (const uint8_t*)p[k + 1];
    if (next < end || next > end + slack) return false;
  }
  return (size_t)((const uint8_t*)p[m - 1] - (const uint8_t*)p[0]) + size[m - 1] <= limit;
}

}  // namespace zb
