// seekable.h — zstd's seekable format (zstd repository, contrib/seekable_format/zstd_seekable_compression_format.md): an
// archive is independent zstd frames back to back from byte 0, followed by a skippable frame that holds the seek table:
//
//   0x184D2A5E  Frame_Size = n * entry + 9  |  n x { Compressed_Size u32, Decompressed_Size u32 [, Checksum u32] }  |
//   Number_Of_Frames u32  Seek_Table_Descriptor u8 (bit 7: checksums; bits 6-2 reserved, 0; bits 1-0 ignored)  0x8F92EAB1
//
// (all little-endian; Checksum = low 32 bits of the XXH64, seed 0, of the frame's content).  This header owns the format:
// cutting an input into frames, the bound, writing the table, parsing and validating it, and turning a content range into
// the frames that cover it.  Pure functions (no CUDA), so that tests/hostsim/seekable.cpp can check them on a CPU; the byte
// writers are also callable from the pack kernel (seekable_kernels.cu).
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <algorithm>
#include <vector>

#if defined(__CUDACC__)
#define SEEK_HD __host__ __device__ inline
#else
#define SEEK_HD inline
#endif

namespace zb {
namespace seek {

constexpr uint32_t SKIPPABLE_MAGIC = 0x184D2A5E, FOOTER_MAGIC = 0x8F92EAB1;
constexpr uint32_t HEADER_BYTES = 8, FOOTER_BYTES = 9;
constexpr uint32_t MIN_ARCHIVE = HEADER_BYTES + FOOTER_BYTES;   // the table frame of an archive of no frames
// the library's result codes (include/zstdb200.h), as (uint32_t)-code
constexpr uint32_t ERR_prefix_unknown = (uint32_t)-10, ERR_corruption_detected = (uint32_t)-20, ERR_srcSize_wrong = (uint32_t)-72;

SEEK_HD uint32_t entry_bytes(bool ck) { return ck ? 12u : 8u; }
SEEK_HD uint64_t table_bytes(uint64_t n, bool ck) { return HEADER_BYTES + n * entry_bytes(ck) + FOOTER_BYTES; }
// Frame_Size (n x entry + 9) is a u32: a writer accepts no more frames than that holds (357 913 940 with checksums, 536 870 910
// without)
inline bool table_fits(uint64_t n, bool ck) { return n <= (0xFFFFFFFFull - FOOTER_BYTES) / entry_bytes(ck); }
SEEK_HD uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
SEEK_HD void st32(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }

// ---- writing ----------------------------------------------------------------------------------------------------------
SEEK_HD void write_header(uint8_t* p, uint64_t n, bool ck) { st32(p, SKIPPABLE_MAGIC); st32(p + 4, (uint32_t)(n * entry_bytes(ck) + FOOTER_BYTES)); }
SEEK_HD void write_entry(uint8_t* p, uint32_t csize, uint32_t dsize, uint32_t cksum, bool ck) {
  st32(p, csize); st32(p + 4, dsize);
  if (ck) st32(p + 8, cksum);
}
SEEK_HD void write_footer(uint8_t* p, uint32_t n, bool ck) { st32(p, n); p[4] = ck ? 0x80 : 0; st32(p + 5, FOOTER_MAGIC); }

// The whole table frame of n frames at out (table_bytes(n, ck) bytes); cksum is read only with ck (and n > 0).
inline void write_table(uint8_t* out, size_t n, const uint32_t* csize, const uint32_t* dsize, const uint32_t* cksum, bool ck) {
  write_header(out, n, ck);
  for (size_t i = 0; i < n; i++) write_entry(out + HEADER_BYTES + i * entry_bytes(ck), csize[i], dsize[i], ck ? cksum[i] : 0, ck);
  write_footer(out + HEADER_BYTES + n * entry_bytes(ck), (uint32_t)n, ck);
}

// ---- cutting the input ------------------------------------------------------------------------------------------------
// Frame i holds bytes [i * fs, min((i + 1) * fs, srcSize)) of the input.
inline uint64_t frame_count(uint64_t srcSize, uint32_t fs) { return (srcSize + fs - 1) / fs; }
inline uint32_t frame_content(uint64_t srcSize, uint32_t fs, uint64_t i) { return (uint32_t)std::min<uint64_t>(fs, srcSize - i * fs); }

// Largest archive of srcSize bytes in frames of fs: every frame at its compress bound (frameBound(content bytes)) and a table
// with checksums.  A destination of this size never overflows, so the pack step needs no overflow path.
template <class FB>
uint64_t bound(uint64_t srcSize, uint32_t fs, FB frameBound) {
  const uint64_t n = frame_count(srcSize, fs);
  uint64_t b = table_bytes(n, true);
  if (n) b += (n - 1) * (uint64_t)frameBound(fs) + frameBound(frame_content(srcSize, fs, n - 1));
  return b;
}

// ---- reading ----------------------------------------------------------------------------------------------------------
struct Footer {
  uint32_t n = 0; bool ck = false;
  uint64_t tableBytes = 0;     // the whole table frame
};

// The last 9 bytes of an archive of srcSize bytes.  0 or an error code:
//   srcSize_wrong        the archive is shorter than 17 bytes, or the table is longer than the archive
//   prefix_unknown       the footer magic is wrong
//   corruption_detected  a reserved bit of the descriptor is set
inline uint32_t parse_footer(const uint8_t* tail, uint64_t srcSize, Footer* f) {
  if (srcSize < MIN_ARCHIVE) return ERR_srcSize_wrong;
  if (rd32(tail + 5) != FOOTER_MAGIC) return ERR_prefix_unknown;
  const uint8_t sfd = tail[4];
  if (sfd & 0x7C) return ERR_corruption_detected;
  f->n = rd32(tail); f->ck = (sfd & 0x80) != 0;
  f->tableBytes = table_bytes(f->n, f->ck);
  if (f->tableBytes > srcSize) return ERR_srcSize_wrong;
  return 0;
}

struct Table {
  uint32_t n = 0; bool ck = false;
  uint64_t tableBytes = 0, dataSize = 0, contentSize = 0;
  uint32_t maxContent = 0, maxCompressed = 0;
  std::vector<uint32_t> csize, dsize, cksum;   // cksum: empty when the table carries none
  std::vector<uint64_t> srcOff, dstOff;        // n + 1 prefix sums of csize / dsize
};

// The table frame (f.tableBytes bytes, the end of an archive of srcSize bytes) after parse_footer.  0 or an error code:
//   prefix_unknown       the skippable magic is wrong
//   corruption_detected  Frame_Size does not match n and the entry size, or the compressed sizes do not add up to exactly
//                        the bytes before the table
inline uint32_t parse_table(const uint8_t* tab, uint64_t srcSize, const Footer& f, Table* t) {
  if (rd32(tab) != SKIPPABLE_MAGIC) return ERR_prefix_unknown;
  if ((uint64_t)rd32(tab + 4) != f.tableBytes - HEADER_BYTES) return ERR_corruption_detected;
  *t = Table();
  t->n = f.n; t->ck = f.ck; t->tableBytes = f.tableBytes;
  t->csize.resize(f.n); t->dsize.resize(f.n); t->srcOff.assign(f.n + 1, 0); t->dstOff.assign(f.n + 1, 0);
  if (f.ck) t->cksum.resize(f.n);
  const uint32_t eb = entry_bytes(f.ck);
  for (uint32_t i = 0; i < f.n; i++) {
    const uint8_t* e = tab + HEADER_BYTES + (uint64_t)i * eb;
    t->csize[i] = rd32(e); t->dsize[i] = rd32(e + 4);
    if (f.ck) t->cksum[i] = rd32(e + 8);
    t->srcOff[i + 1] = t->srcOff[i] + t->csize[i]; t->dstOff[i + 1] = t->dstOff[i] + t->dsize[i];
    t->maxCompressed = std::max(t->maxCompressed, t->csize[i]); t->maxContent = std::max(t->maxContent, t->dsize[i]);
  }
  t->dataSize = srcSize - f.tableBytes;
  if (t->srcOff[f.n] != t->dataSize) return ERR_corruption_detected;
  t->contentSize = t->dstOff[f.n];
  return 0;
}

// Both steps over an archive in host memory.
inline uint32_t parse(const uint8_t* src, uint64_t srcSize, Table* t) {
  Footer f;
  if (!src && srcSize) return ERR_srcSize_wrong;
  if (uint32_t r = parse_footer(src + srcSize - (srcSize >= FOOTER_BYTES ? FOOTER_BYTES : srcSize), srcSize, &f)) return r;
  return parse_table(src + srcSize - f.tableBytes, srcSize, f, t);
}

// ---- range plan -------------------------------------------------------------------------------------------------------
// One frame that overlaps content bytes [offset, offset + length): it is src[srcOff .. + csize) and decodes to dsize bytes,
// of which [skip, skip + take) are in the range and go to dst[dstOff ..).  A frame with skip > 0 or take < dsize is an edge
// frame (the first and the last): it decodes into scratch and its in-range part is copied out; the others decode in place.
struct Piece {
  uint32_t frame; uint32_t csize, dsize; uint64_t srcOff, dstOff; uint32_t skip, take;
  bool edge() const { return skip != 0 || take != dsize; }
};

// The frames that cover content bytes [offset, offset + length), in archive order.  Frames of no content are never chosen.
// 0, or srcSize_wrong when the range ends past the content (nothing is chosen).
inline uint32_t plan_range(const Table& t, uint64_t offset, uint64_t length, std::vector<Piece>* out) {
  out->clear();
  if (offset > t.contentSize || length > t.contentSize - offset) return ERR_srcSize_wrong;
  if (length == 0) return 0;
  const uint64_t end = offset + length;
  // first frame whose content ends after offset
  uint32_t i = (uint32_t)(std::upper_bound(t.dstOff.begin() + 1, t.dstOff.end(), offset) - (t.dstOff.begin() + 1));
  for (; i < t.n && t.dstOff[i] < end; i++) {
    if (t.dsize[i] == 0) continue;
    const uint64_t lo = std::max(offset, t.dstOff[i]), hi = std::min(end, t.dstOff[i + 1]);
    out->push_back({i, t.csize[i], t.dsize[i], t.srcOff[i], lo - offset, (uint32_t)(lo - t.dstOff[i]), (uint32_t)(hi - lo)});
  }
  return 0;
}

}  // namespace seek
}  // namespace zb
