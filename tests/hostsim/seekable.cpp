// C entry points over zstandard_b200/csrc/seekable.h (g++, no CUDA) for tests/test_seekable.py: the table writer, the
// parser and the range planner.
#include <string.h>

#include "../../zstandard_b200/csrc/seekable.h"

using namespace zb::seek;

extern "C" {

uint64_t sk_table_bytes(uint64_t n, int ck) { return table_bytes(n, ck != 0); }
int sk_table_fits(uint64_t n, int ck) { return table_fits(n, ck != 0); }

void sk_write_table(uint8_t* out, size_t n, const uint32_t* csize, const uint32_t* dsize, const uint32_t* cksum, int ck) {
  write_table(out, n, csize, dsize, cksum, ck != 0);
}

// fields: [n, ck, tableBytes, dataSize, contentSize, maxContent, maxCompressed]; entries: n x (csize, dsize, cksum) when
// non-null.  Returns 0 or the error code.
uint32_t sk_parse(const uint8_t* src, uint64_t size, uint64_t* fields, uint32_t* entries) {
  Table t;
  const uint32_t r = parse(src, size, &t);
  if (r) return r;
  const uint64_t f[7] = {t.n, t.ck, t.tableBytes, t.dataSize, t.contentSize, t.maxContent, t.maxCompressed};
  memcpy(fields, f, sizeof f);
  for (uint32_t i = 0; entries && i < t.n; i++) {
    entries[3 * i] = t.csize[i]; entries[3 * i + 1] = t.dsize[i]; entries[3 * i + 2] = t.ck ? t.cksum[i] : 0;
  }
  return 0;
}

// The plan of [offset, offset + length) over the archive: per piece (frame, dstOff, skip, take, srcOff, csize).  *count = the
// number of pieces; returns 0 or the error code.
uint32_t sk_plan(const uint8_t* src, uint64_t size, uint64_t offset, uint64_t length, uint64_t* out, uint64_t* count) {
  Table t;
  uint32_t r = parse(src, size, &t);
  std::vector<Piece> p;
  if (!r) r = plan_range(t, offset, length, &p);
  *count = p.size();
  for (size_t k = 0; k < p.size(); k++) {
    uint64_t* o = out + 6 * k;
    o[0] = p[k].frame; o[1] = p[k].dstOff; o[2] = p[k].skip; o[3] = p[k].take; o[4] = p[k].srcOff; o[5] = p[k].csize;
  }
  return r;
}

}  // extern "C"
