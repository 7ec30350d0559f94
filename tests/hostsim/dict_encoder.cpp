// tests/hostsim/dict_encoder.cpp — CPU emulation of the GPU encoder with the context's dictionary (TEST AID ONLY).
//
// What zstdb200_compress*_using_dict runs on the device, restated for g++: the lock-step emulation of
// k_enc_match<DFAST, true> (the warp-parallel match finder of hostsim.cpp with the dictionary's match tables, offsets into
// its content and its repeat offsets) and the serial statement of k_enc_entropy<true> (serial_encoder.h's section writers with
// the Dictionary_ID field and, in a frame's first block, the dictionary's Huffman / FSE tables where they are cheaper).  The
// dictionary is prepared by the library's own enc_dict_prepare (zb_encode.cuh) over the decoder's dict_load, so the emulation
// and the kernels start from the same tables.  tests/test_dictionary_compress.py builds this file into its own library and
// compares it with the oracle, libzstd and (on a GPU) the kernels' bytes.  It is never linked into libzstdb200.so.
#include <stdio.h>
#include <stdlib.h>
#include <algorithm>
#include <cstring>
#include <vector>
#include "../../zstandard_b200/csrc/zb_encode.cuh"
#include "serial_encoder.h"

using namespace zb;

namespace {

// the dictionary (hsdict_set): the decoder's parse and the encoder's prepared block
DictState g_ds; std::vector<u8> g_bytes, g_enc; bool g_have = false;

// literals section (DecodeLiteralsBlock ZStdDecompress.cs:683-821).  Returns bytes written (0 = no room).
// ed: the dictionary when this is the first block of a frame compressed with an entropy dictionary (treeless literals), else null.
u32 enc_literals_d(u8* out, u32 cap, const u8* lits, u32 n, u16* stateScratch, u8* symScratch, const EncDict* ed) {
  auto raw = [&]() -> u32 {
    const u32 lh = n < 32 ? 1 : (n < 4096 ? 2 : 3);
    if (lh + n > cap) return 0;
    if (lh == 1) out[0] = (u8)(n << 3); else if (lh == 2) { u32 v = (1u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); }
    else { u32 v = (3u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); }
    for (u32 i = 0; i < n; i++) out[lh + i] = lits[i];
    return lh + n;
  };
  if (n < 64) return raw();
  u32 count[256]; for (u32 i = 0; i < 256; i++) count[i] = 0;
  for (u32 i = 0; i < n; i++) count[lits[i]]++;
  u32 maxSym = 255; while (maxSym > 0 && !count[maxSym]) maxSym--;
  u32 largest = 0; for (u32 s = 0; s <= maxSym; s++) if (count[s] > largest) largest = count[s];
  if (largest == n) {   // rle literals
    const u32 lh = n < 32 ? 1 : (n < 4096 ? 2 : 3);
    if (lh + 1 > cap) return 0;
    if (lh == 1) out[0] = (u8)(1 | (n << 3)); else if (lh == 2) { u32 v = 1 | (1u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); }
    else { u32 v = 1 | (3u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); }
    out[lh] = lits[0];
    return lh + 1;
  }
  if (largest <= (n >> 7) + 4) return raw();   // too flat to be worth it
  HufEnc he; HufBuildScratch hsc;
  u32 maxBits = fse_optimal_log(11, n, maxSym, 1); if (maxBits > 11) maxBits = 11;
  if (!huf_build(he, count, maxSym, maxBits, hsc)) return raw();
  const bool single = n < 256;
  const u32 lhSize = 3 + (n >= 1024) + (n >= 16384);
  if (lhSize + 8 > cap) return 0;
  u8* body = out + lhSize; const u32 bodyCap = cap - lhSize;
  u32 hdr = huf_write_header(body, bodyCap, he, stateScratch, symScratch);
  if (!hdr) return raw();
  const bool treeless = ed && huf_dict_better(ed->huf, he, hdr, count);
  const HufEnc& code = treeless ? ed->huf : he;
  u32 csize = treeless ? 0 : hdr;
  if (single) {
    u32 s = huf_encode_stream(body + csize, bodyCap - csize, lits, n, code);
    if (!s) return raw();
    csize += s;
  } else {
    const u32 seg = (n + 3) / 4;
    if (csize + 6 > bodyCap) return raw();
    u8* jump = body + csize; csize += 6;
    for (u32 k = 0; k < 4; k++) {
      const u32 from = k * seg, len = k < 3 ? seg : n - 3 * seg;
      u32 s = huf_encode_stream(body + csize, bodyCap - csize, lits + from, len, code);
      if (!s || s > 65535) return raw();
      if (k < 3) { jump[2 * k] = (u8)s; jump[2 * k + 1] = (u8)(s >> 8); }
      csize += s;
    }
  }
  const u32 minGain = (n >> 6) + 2;
  if (csize + minGain >= n) return raw();
  // header: type 2 (compressed) or 3 (treeless: the dictionary's code), size format by lhSize
  const u32 lt = treeless ? 3 : 2;
  if (lhSize == 3) { u32 v = lt | ((single ? 0u : 1u) << 2) | (n << 4) | (csize << 14); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); }
  else if (lhSize == 4) { u32 v = lt | (2u << 2) | (n << 4) | (csize << 18); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); out[3] = (u8)(v >> 24); }
  else { u32 v = lt | (3u << 2) | (n << 4) | (csize << 22); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); out[3] = (u8)(v >> 24); out[4] = (u8)(csize >> 10); }
  return lhSize + csize;
}

u32 enc_seq_table_d(FseCTable& ct, u16* stateTable, u8* symScratch, const u8* codes, u32 nbSeq, const SeqKind& k, int level,
                        u8* out, u32 cap, u32* used, const EncDict* ed, int kind) {
  u32 count[53]; for (u32 i = 0; i <= k.maxSym; i++) count[i] = 0;
  for (u32 i = 0; i < nbSeq; i++) count[codes[i]]++;
  return enc_seq_table_counts_dict(ct, stateTable, symScratch, count, codes[nbSeq - 1], nbSeq, k, level, out, cap, used, ed, kind);
}

// Returns bytes written, 0 on failure (caller falls back to a raw block).  ed: as for enc_literals (repeat-mode tables).
u32 enc_sequences_d(u8* out, u32 cap, const SeqStore& st, u8* codes, u16* ctables, u8* symScratch, int level, const EncDict* ed) {
  const u32 nbSeq = st.n;
  if (cap < 4) return 0;
  u32 op = enc_seq_count_header(out, nbSeq);
  if (nbSeq == 0) return op;
  u8 *llc = codes, *ofc = codes + st.cap, *mlc = codes + 2 * st.cap;
  for (u32 i = 0; i < nbSeq; i++) {
    u32 ll, ob, mlm3; seq_get(st, i, ll, ob, mlm3);
    llc[i] = (u8)ll_code(ll); ofc[i] = (u8)highbit(ob); mlc[i] = (u8)ml_code(mlm3);
  }
  const SeqKind kLL = seq_kind(KIND_LL), kOF = seq_kind(KIND_OF), kML = seq_kind(KIND_ML);
  u8* modeByte = out + op++; u32 used;
  FseCTable ctLL, ctOF, ctML;
  const u32 mLL = enc_seq_table_d(ctLL, ctables, symScratch, llc, nbSeq, kLL, level, out + op, cap - op, &used, ed, KIND_LL); if (mLL == 0xFF) return 0; op += used;
  const u32 mOF = enc_seq_table_d(ctOF, ctables + 514, symScratch, ofc, nbSeq, kOF, level, out + op, cap - op, &used, ed, KIND_OF); if (mOF == 0xFF) return 0; op += used;
  const u32 mML = enc_seq_table_d(ctML, ctables + 1028, symScratch, mlc, nbSeq, kML, level, out + op, cap - op, &used, ed, KIND_ML); if (mML == 0xFF) return 0; op += used;
  *modeByte = (u8)((mLL << 6) | (mOF << 4) | (mML << 2));
  u8* e = enc_seq_bitstream(out + op, out + cap, st, llc, ofc, mlc, ctLL, ctOF, ctML);
  if (!e) return 0;
  return (u32)(e - out);
}

// frame assembly: serial_encoder.h's encode_frame_with with the dictionary.
// ed: the encoder dictionary (null: none).  Its id goes into the header (none for a raw-content dictionary, id 0); the first
// block may code with its entropy tables.
template <class BlockSeqs>
u32 encode_frame_d(const u8* src, u32 size, u8* dst, u32 cap, int level, int checksum, u8* codes, u16* ctables, u8* symScratch,
                 BlockSeqs& blockSeqs, const EncDict* ed) {
  u32 op = 0;
  const u32 dictID = ed ? ed->dictID : 0;
  const u32 fhs = enc_frame_header_size(size, dictID);
  if (cap < fhs + 3 + (checksum ? 4 : 0)) return zerr(ZE_dstSize_tooSmall);
  op = enc_frame_header(dst, size, checksum, dictID);                 // single segment
  const u32 tail = checksum ? 4 : 0;
  u32 pos = 0, blk = 0;
  do {
    const u32 bsize = size - pos < BLOCKSIZE_MAX ? size - pos : BLOCKSIZE_MAX;
    const u32 last = pos + bsize == size;
    const u8* bstart = src + pos;
    if (op + 3 + tail > cap) return zerr(ZE_dstSize_tooSmall);
    bool rle = bsize > 0;
    for (u32 i = 1; i < bsize && rle; i++) if (bstart[i] != bstart[0]) rle = false;
    SeqStore st; st.n = 0; st.nlits = 0; st.seqs = nullptr; st.lits = nullptr; st.cap = 0;
    const bool haveSeqs = blockSeqs(st, blk, bstart, bsize, rle && bsize >= 2);   // always called: keeps matcher state in step
    if (rle && bsize >= 2) {
      if (op + 4 + tail > cap) return zerr(ZE_dstSize_tooSmall);
      const u32 h = last | (1u << 1) | (bsize << 3);
      dst[op] = (u8)h; dst[op + 1] = (u8)(h >> 8); dst[op + 2] = (u8)(h >> 16); dst[op + 3] = bstart[0]; op += 4;
    } else {
      u32 csize = 0; bool compressed = false;
      if (haveSeqs) {
        u32 room = bsize - 1 < BLOCKSIZE_MAX - 1 ? bsize - 1 : BLOCKSIZE_MAX - 1;   // must beat raw and stay < 128 KiB (:1880)
        const u32 avail = cap - op - 3 - tail;
        if (room > avail) room = avail;
        u8* body = dst + op + 3;
        const EncDict* const edb = ed && ed->hasEntropy && blk == 0 ? ed : nullptr;   // only the first block's "previous tables" are the dictionary's
        const u32 l = enc_literals_d(body, room, st.lits, st.nlits, ctables, symScratch, edb);
        if (l) {
          const u32 s = enc_sequences_d(body + l, room - l, st, codes, ctables, symScratch, level, edb);
          if (s && l + s < bsize) { csize = l + s; compressed = true; }
        }
        blockSeqs.done(compressed);
      }
      if (compressed) {
        const u32 h = last | (2u << 1) | (csize << 3);
        dst[op] = (u8)h; dst[op + 1] = (u8)(h >> 8); dst[op + 2] = (u8)(h >> 16); op += 3 + csize;
      } else {
        if (op + 3 + bsize + tail > cap) return zerr(ZE_dstSize_tooSmall);
        const u32 h = last | (0u << 1) | (bsize << 3);
        dst[op] = (u8)h; dst[op + 1] = (u8)(h >> 8); dst[op + 2] = (u8)(h >> 16); op += 3;
        for (u32 i = 0; i < bsize; i++) dst[op + i] = bstart[i];
        op += bsize;
      }
    }
    pos += bsize; blk++;
  } while (pos < size);
  return op;
}

// lock-step emulation of k_enc_match<DFAST, true>: hostsim.cpp's WarpMatcher with the dictionary's tables
struct DictWarpMatcher {
  std::vector<u16> tab; u32 hlogL, hlogS, mls; bool dfast;
  const u8* src; u32 size; u32 rep1 = 1, rep2 = 4;   // (the dictionary's rep[0], rep[1] when there is one)
  std::vector<u32> seqs; std::vector<u8> lits;
  const EncDict* ed = nullptr;     // the dictionary (k_enc_match<DFAST, true>), null: none
  static u32 h64(u64 v, u32 hlog, u32 mls) { return hash64(v, hlog, mls); }
  static bool candFrom(u32 p, u32 e, u32& c) { u32 d = (p - e) & 0xFFFF; if (!d) d = 0x10000; c = p - d; return d <= p; }
  u32 extend(u32 a, u32 off, u32 end) { u32 n = 0; while (a + n < end && src[a + n] == src[a + n - off]) n++; return n; }
  bool operator()(SeqStore& st, u32 blk, const u8* bstart, u32 bsize, bool isRle) {
    if (isRle || bsize < 64) return false;
    seqs.assign(2 * (BLOCKSIZE_MAX / 4 + 64), 0); lits.assign(BLOCKSIZE_MAX + 64, 0);
    u32 nseq = 0, nlits = 0;
    const u32 bpos = (u32)(bstart - src), bend = bpos + bsize;
    if (blk > 0) { rep1 = 0; rep2 = 0; }
    u16* tabL = tab.data(); u16* tabS = tab.data() + (1u << hlogL);
    {
      // every block is an independent unit of the match kernel: cleared tables, primed with the 16 KiB before the block
      std::fill(tab.begin(), tab.end(), (u16)0);
      const u32 b0 = (u32)(bstart - src);
      if (blk > 0) for (u32 q = b0 - 16384u; q < b0; q++) {        // ascending: the last position of a hash value is the one kept
        const u64 v = ld64(src + q);
        tabL[h64(v, hlogL, dfast ? 8 : mls)] = (u16)q; if (dfast) tabS[h64(v, hlogS, mls)] = (u16)q;
      }
    }
    u32 anchor = bpos; const u32 ilimit = bend - 8; u32 p0 = bpos + (bpos == 0 ? 1 : 0);
    while (p0 < ilimit) {
      const u32 step = 1 + ((p0 - anchor) >> 8);
      u32 p[32], hL[32], hS[32], candL[32], candS[32]; bool act[32], vL[32], vS[32], okL[32], okS[32], rok[32]; u64 v[32];
      for (u32 l = 0; l < 32; l++) {
        p[l] = p0 + l * step; act[l] = p[l] < ilimit; v[l] = act[l] ? ld64(src + p[l]) : 0;
        hL[l] = act[l] ? h64(v[l], hlogL, dfast ? 8 : mls) : (0x80000000u | l);
        hS[l] = act[l] ? h64(v[l], hlogS, mls) : (0x80000000u | l);
      }
      for (u32 l = 0; l < 32; l++) {
        i32 low = -1; for (i32 k = (i32)l - 1; k >= 0; k--) if (hL[k] == hL[l]) { low = k; break; }
        if (low >= 0) { candL[l] = p[low]; vL[l] = act[l]; } else vL[l] = act[l] && candFrom(p[l], tabL[hL[l] & 0xFFFFFF], candL[l]);
        vS[l] = false;
        if (dfast) { low = -1; for (i32 k = (i32)l - 1; k >= 0; k--) if (hS[k] == hS[l]) { low = k; break; }
          if (low >= 0) { candS[l] = p[low]; vS[l] = act[l]; } else vS[l] = act[l] && candFrom(p[l], tabS[hS[l] & 0xFFFFFF], candS[l]); }
      }
      i32 fl = -1;
      u32 candDL[32], candDS[32]; bool okDL[32], okDS[32];
      const u8* const dc = ed ? enc_dict_content(ed) : nullptr;
      for (u32 l = 0; l < 32; l++) {
        okL[l] = vL[l] && (dfast ? ld64(src + candL[l]) == v[l] : ld32(src + candL[l]) == (u32)v[l]);
        okS[l] = dfast && vS[l] && ld32(src + candS[l]) == (u32)v[l];
        okDL[l] = okDS[l] = false;                                    // dictionary: chunk long, dict long, chunk short, dict short
        if (ed && act[l] && !okL[l]) {
          candDL[l] = enc_dict_table(ed, dfast ? EDT_LONG : (mls == 6 ? EDT_MLS6 : EDT_MLS5))[hash64(v[l], ENC_DICT_HLOG, dfast ? 8 : mls)];
          if (candDL[l] != ENC_DICT_EMPTY) okDL[l] = dfast ? ld64(dc + candDL[l]) == v[l] : ld32(dc + candDL[l]) == (u32)v[l];
        }
        if (ed && dfast && act[l] && !okL[l] && !okDL[l] && !okS[l]) {
          candDS[l] = enc_dict_table(ed, EDT_MLS5)[hash64(v[l], ENC_DICT_HLOG, mls)];
          if (candDS[l] != ENC_DICT_EMPTY) okDS[l] = ld32(dc + candDS[l]) == (u32)v[l];
        }
        rok[l] = act[l] && rep1 != 0 && rep1 <= p[l] && ld32(src + p[l] - rep1) == (u32)v[l];
        if (fl < 0 && (okL[l] || okS[l] || okDL[l] || okDS[l] || rok[l])) fl = (i32)l;
      }
      // a repeat-offset match a few bytes further on beats a table match here (cheaper to code)
      if (fl >= 0 && !rok[fl]) { const int look = 3; for (i32 l = fl + 1; l <= fl + look && l < 32; l++) if (rok[l]) { fl = l; break; } }
      auto insert = [&](u32 limit) {   // ascending lanes: last writer wins; nothing at or beyond the restart position
        for (u32 l = 0; l < 32; l++) if (act[l] && p[l] < limit) { tabL[hL[l]] = (u16)p[l]; if (dfast) tabS[hS[l]] = (u16)p[l]; } };
      if (fl < 0) { insert(0xFFFFFFFFu); p0 += 32 * step; continue; }
      u32 pos = p[fl]; const u32 kind = rok[fl] ? 0 : (okL[fl] ? 1 : (okDL[fl] ? 3 : (okS[fl] ? 2 : 4)));
      u32 cnd = kind == 0 ? pos - rep1 : (kind == 1 ? candL[fl] : (kind == 3 ? candDL[fl] : (kind == 4 ? candDS[fl] : candS[fl])));
      u32 off, mlen;
      if (kind >= 3) {                                                 // against the dictionary content, up to its end
        const u32 dsize = ed->contentSize; off = pos + (dsize - cnd);
        const u32 fend = std::min(bend, pos + (dsize - cnd));
        mlen = 4; while (pos + mlen < fend && src[pos + mlen] == dc[cnd + mlen]) mlen++;
        while (pos > anchor && cnd > 0 && src[pos - 1] == dc[cnd - 1]) { pos--; cnd--; mlen++; }
      } else {
        off = pos - cnd;
        mlen = 4 + extend(pos + 4, off, bend);
        while (pos > anchor && cnd > 0 && src[pos - 1] == src[cnd - 1]) { pos--; cnd--; mlen++; }
      }
      insert(pos + mlen);
      const u32 ll = pos - anchor; u32 offBase;
      if (kind == 0 && ll > 0) offBase = 1; else { offBase = off + 3; rep2 = rep1; rep1 = off; }
      memcpy(lits.data() + nlits, src + anchor, ll);
      seqs[2 * nseq] = (ll & 0xFFFF) | (((mlen - 3) & 0xFFFF) << 16);
      seqs[2 * nseq + 1] = (offBase & 0x3FFFFFFFu) | ((((mlen - 3) >> 16) & 1) << 30) | (((ll >> 16) & 1) << 31);
      nlits += ll; nseq++;
      anchor = pos + mlen; p0 = anchor;
      if (p0 <= ilimit) {

        while (rep2 != 0 && rep2 <= p0 && p0 <= ilimit && ld32(src + p0) == ld32(src + p0 - rep2)) {
          const u32 rlen = 4 + extend(p0 + 4, rep2, bend);
          std::swap(rep1, rep2);
          tabL[h64(ld64(src + p0), hlogL, dfast ? 8 : mls)] = (u16)p0; if (dfast) tabS[h64(ld64(src + p0), hlogS, mls)] = (u16)p0;
          seqs[2 * nseq] = ((rlen - 3) & 0xFFFF) << 16; seqs[2 * nseq + 1] = 1u | ((((rlen - 3) >> 16) & 1) << 30);
          nseq++; p0 += rlen; anchor = p0;
        }
      }
    }
    const u32 ll = bend - anchor; memcpy(lits.data() + nlits, src + anchor, ll); nlits += ll;
    st.seqs = seqs.data(); st.n = nseq; st.cap = BLOCKSIZE_MAX / 4 + 64; st.lits = lits.data(); st.nlits = nlits;
    return true;
  }
  void done(bool) {}
};

uint32_t compress(uint8_t* dst, uint32_t cap, const uint8_t* src_in, uint32_t size, int level, int checksum, uint32_t batch_max, const EncDict* ed) {
  if (ed->err) return zerr(ed->err);
  std::vector<u8> padded(size + 64, 0);
  u8* src = padded.data() + 16;
  if (size) memcpy(src, src_in, size);
  const bool big = batch_max > BLOCKSIZE_MAX;
  DictWarpMatcher m; m.src = src; m.size = size; m.dfast = level >= 3; m.hlogL = enc_hlog_long(level, big); m.hlogS = enc_hlog_short(level, big); m.mls = level <= 1 ? 6 : 5;
  m.tab.assign((1u << m.hlogL) + (1u << m.hlogS), 0);
  m.ed = ed; m.rep1 = ed->rep[0]; m.rep2 = ed->rep[1];
  const u32 seqCap = BLOCKSIZE_MAX / 4 + 64;
  std::vector<u8> codes(3 * seqCap), sym(4096); std::vector<u16> ct(3 * 514 + 16);
  return encode_frame_d(src, size, dst, cap, level, checksum, codes.data(), ct.data(), sym.data(), m, ed);
}

}  // namespace

// The dictionary of the emulation (the device's zstdb200_load_dictionary); size 0 removes it.
extern "C" void hsdict_set(const uint8_t* dict, uint32_t size) {
  g_have = false;
  if (!dict || size == 0) return;
  g_bytes.assign(dict, dict + size); g_bytes.resize(size + 64, 0);
  static HufBuildWk wk; static HufFseScratch fs; static u8 slot[260], tableSymbol[512]; static s16 norm[64]; static u16 next[64];
  dict_load(g_bytes.data(), size, g_ds, wk, fs, slot, norm, next);
  g_enc.assign(enc_dict_bytes(g_ds.err ? 0 : g_ds.contentSize), 0);
  enc_dict_prepare(g_bytes.data(), size, g_ds, reinterpret_cast<EncDict*>(g_enc.data()), wk, fs, slot, tableSymbol);
  g_have = true;
}
// where the loaded dictionary's content starts (its three repeat offsets are the 12 bytes before it)
extern "C" uint32_t hsdict_content_offset() { return g_have ? g_ds.contentOff : 0; }
// One frame as zstdb200_compress_batch_using_dict writes it (the checksum slot left for the caller, as k_enc_xxh fills it);
// batch_max: the largest chunk of the call (the match stage's table sizes).  GENERIC without a dictionary, dictionary_corrupted
// for a malformed one.
extern "C" uint32_t hsdict_compress(uint8_t* dst, uint32_t cap, const uint8_t* src, uint32_t size, int level, int checksum, uint32_t batch_max) {
  if (!g_have) return zerr(ZE_GENERIC);
  return compress(dst, cap, src, size, level, checksum, batch_max, reinterpret_cast<const EncDict*>(g_enc.data()));
}
