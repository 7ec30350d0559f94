// C entry points over zstandard_b200/csrc/host_plan.h (g++, no CUDA) for tests/test_host_plan.py.  Ranges come back as
// (lo, hi) pairs in `out`; every function returns how many it wrote.
#include <vector>

#include "../../zstandard_b200/csrc/host_plan.h"

using namespace zb;

static size_t put(const std::vector<Range>& r, uint64_t* out) {
  for (size_t k = 0; k < r.size(); k++) { out[2 * k] = r[k].lo; out[2 * k + 1] = r[k].hi; }
  return r.size();
}

extern "C" {

size_t hp_subbatches(size_t n, size_t maxIn, size_t maxOut, size_t maxItems, const uint32_t* in, const uint32_t* outBytes,
                     uint64_t* out, int* tooBig) {
  bool big = false;
  const size_t k = put(make_subbatches(n, maxIn, maxOut, maxItems, [&](size_t i) { return (size_t)in[i]; },
                                       [&](size_t i) { return (size_t)outBytes[i]; }, &big), out);
  *tooBig = big;
  return k;
}

// cost(i) = in[i] + outBytes[i] + 1, as run_host_batch computes it
size_t hp_split(const uint64_t* ranges, size_t nr, size_t nd, const uint32_t* in, const uint32_t* outBytes, uint64_t* out) {
  std::vector<Range> subs;
  for (size_t k = 0; k < nr; k++) subs.push_back({(size_t)ranges[2 * k], (size_t)ranges[2 * k + 1]});
  return put(split_over_devices(subs, nd, [&](size_t i) { return (uint64_t)in[i] + outBytes[i] + 1; }), out);
}

size_t hp_slices(const uint32_t* srcSize, const uint32_t* dstCap, size_t m, int decode, size_t sliceBytes, uint64_t* out) {
  return put(plan_slices(srcSize, dstCap, m, decode != 0, sliceBytes), out);
}

int hp_back_to_back(const uint64_t* addr, const uint32_t* size, size_t m, size_t slack, size_t limit) {
  std::vector<const void*> p(m);
  for (size_t k = 0; k < m; k++) p[k] = (const void*)(uintptr_t)addr[k];
  return back_to_back(p.data(), size, m, slack, limit);
}

// byte offsets of the four arrays of DescView(base, m) from base, and DescView::bytes(m)
void hp_desc_layout(size_t m, uint64_t* out) {
  std::vector<uint64_t> buf(3 * m + 1);
  unsigned char* base = (unsigned char*)buf.data();
  const DescView v(base, m);
  out[0] = (unsigned char*)v.srcOff - base; out[1] = (unsigned char*)v.dstOff - base;
  out[2] = (unsigned char*)v.srcSize - base; out[3] = (unsigned char*)v.dstCap - base; out[4] = DescView::bytes(m);
}

size_t hp_min_slice_items(int decode) { return decode ? MIN_SLICE_ITEMS_DECODE : MIN_SLICE_ITEMS_ENCODE; }

}  // extern "C"
