// enc_sections.cpp — CPU twin of tests/gpu_harness/enc_sections.cu: the serial section writers of serial_encoder.h (enc_literals,
// enc_sequences) on the same case layout, plus the Huffman / FSE primitives and code tables of zb_encode.cuh on caller data, for
// tests/test_encoder_sections.py.
#include <cstring>
#include <vector>
#include "../../zstandard_b200/csrc/zb_encode.cuh"
#include "serial_encoder.h"

using namespace zb;

namespace {
// raw literals section, as warp_enc_literals writes it at the negative levels; 0 = no room
u32 raw_literals(u8* out, u32 cap, const u8* lits, u32 n) {
  const u32 lh = n < 32 ? 1 : (n < 4096 ? 2 : 3);
  if (lh + n > cap) return 0;
  if (lh == 1) out[0] = (u8)(n << 3); else if (lh == 2) { const u32 v = (1u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); }
  else { const u32 v = (3u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); }
  memcpy(out + lh, lits, n);
  return lh + n;
}
}  // namespace

// Same descriptor layout and in-place output as enc_sections_run (tests/gpu_harness/enc_sections.cu).
extern "C" void es_run(uint32_t n, const uint64_t* desc, const uint8_t* lits, const uint32_t* seqs, uint8_t* out, uint32_t* sizes) {
  const u32 seqCap = BLOCKSIZE_MAX / 4 + 64;
  std::vector<u8> codes(3 * seqCap), sym(4096); std::vector<u16> ct(3 * 514 + 16);
  for (u32 c = 0; c < n; c++) {
    const uint64_t* d = desc + 8 * (size_t)c;
    SeqStore st;
    st.lits = const_cast<u8*>(lits + d[0]); st.nlits = (u32)d[1];
    st.seqs = const_cast<u32*>(seqs + d[2]); st.n = (u32)d[3]; st.cap = seqCap;
    const int level = (int)(int64_t)d[4];
    const u32 cap = (u32)d[5];
    u8* const body = out + d[6] + 64 + d[7];
    const u32 l = level < 0 ? raw_literals(body, cap, st.lits, st.nlits) : enc_literals(body, cap, st.lits, st.nlits, ct.data(), sym.data());
    u32 s = 0;
    if (l) s = enc_sequences(body + l, cap - l, st, codes.data(), ct.data(), sym.data(), level);
    sizes[2 * c] = l; sizes[2 * c + 1] = s;
  }
}

// huf_sort_symbols + huf_build_sorted on count[0..255] with the length limit maxBits; nbBits / weight: 256 entries each.
// Returns 0 when no code was built, else 1 (tableLog in *tl).  hdr: huf_write_header's output (hdrCap bytes), its size in *hdrSize.
extern "C" int es_huf(const uint32_t* count, uint32_t maxBits, uint8_t* nbBits, uint8_t* weight, uint32_t* tl, uint8_t* hdr, uint32_t hdrCap,
                      uint32_t* hdrSize) {
  static HufEnc he; static HufBuildScratch sc; u16 state[512 + 16]; u8 sym[512 + 16];
  u32 maxSym = 255; while (maxSym > 0 && !count[maxSym]) maxSym--;
  const u32 n = huf_sort_symbols(sc.order, count, maxSym);
  if (!huf_build_sorted(he, count, n, maxBits, sc)) return 0;
  for (u32 s = 0; s < 256; s++) { nbBits[s] = he.code[s].nbBits; weight[s] = he.weight[s]; }
  *tl = he.tableLog;
  *hdrSize = huf_write_header(hdr, hdrCap, he, state, sym);
  return 1;
}

extern "C" uint32_t es_fse_optimal_log(uint32_t maxLog, uint32_t total, uint32_t maxSym, uint32_t minus) {
  return fse_optimal_log(maxLog, total, maxSym, minus);
}

extern "C" int es_fse_normalize(int16_t* norm, uint32_t tableLog, const uint32_t* count, uint32_t total, uint32_t maxSym) {
  return fse_normalize(norm, tableLog, count, total, maxSym) ? 1 : 0;
}

extern "C" uint32_t es_fse_write_ncount(uint8_t* out, uint32_t cap, const int16_t* norm, uint32_t maxSym, uint32_t tableLog) {
  return fse_write_ncount(out, cap, norm, maxSym, tableLog);
}

// ll_code / ml_code of v[0..n) (ml_code takes matchLength - 3), and enc_seq_count_header of v[i] into hdr[3 i..] (length in hlen[i])
extern "C" void es_codes(uint32_t n, const uint32_t* v, uint32_t* ll, uint32_t* ml, uint8_t* hdr, uint32_t* hlen) {
  for (u32 i = 0; i < n; i++) { ll[i] = ll_code(v[i]); ml[i] = ml_code(v[i]); hlen[i] = enc_seq_count_header(hdr + 3 * (size_t)i, v[i]); }
}
