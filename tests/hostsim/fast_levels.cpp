// tests/hostsim/fast_levels.cpp — CPU emulation of the GPU encoder at the negative levels -7..-1 (TEST AID ONLY).
//
// What the compress calls run on the device for level -a, restated for g++: the lock-step emulation of k_enc_match<false, DICT,
// true> (libzstd's fast loop: lanes 2k and 2k + 1 probe k * step and k * step + 1, step = 1 + a growing over long runs without a
// match; per pair the repeat offset at the next pair's start, then the table at 2k, then at 2k + 1; after a match libzstd's
// table fill at current0 + 2 and at the match end - 2) and the serial statement of k_enc_entropy at those levels (literals always
// raw, sequences as at level 1, the dictionary's repeat-mode tables allowed in a frame's first block).  With the dictionary of
// hsdict_set the matcher also looks up the dictionary's match table, as dict_encoder.cpp's emulation of the dictionary kernels
// does; that file is included for the dictionary's preparation and the sequence section writer.  tests/test_fast_levels.py
// builds this file into its own library.  It is never linked into libzstdb200.so.
#include "dict_encoder.cpp"

namespace {

struct FastWarpMatcher {
  std::vector<u16> tab; u32 hlog, mls, accel;
  const u8* src; u32 rep1, rep2;
  std::vector<u32> seqs; std::vector<u8> lits;
  const EncDict* ed = nullptr;     // the dictionary (k_enc_match<false, true, true>), null: none
  static bool candFrom(u32 p, u32 e, u32& c) { u32 d = (p - e) & 0xFFFF; if (!d) d = 0x10000; c = p - d; return d <= p; }
  u32 extend(u32 a, u32 off, u32 end) { u32 n = 0; while (a + n < end && src[a + n] == src[a + n - off]) n++; return n; }
  bool operator()(SeqStore& st, u32 blk, const u8* bstart, u32 bsize, bool isRle) {
    if (isRle || bsize < 64) return false;
    seqs.assign(2 * (BLOCKSIZE_MAX / 4 + 64), 0); lits.assign(BLOCKSIZE_MAX + 64, 0);
    u32 nseq = 0, nlits = 0;
    const u32 bpos = (u32)(bstart - src), bend = bpos + bsize;
    if (blk > 0) { rep1 = 0; rep2 = 0; }
    u16* const t = tab.data();
    std::fill(tab.begin(), tab.end(), (u16)0);                      // every block is an independent unit of the match kernel,
    if (blk > 0) for (u32 q = bpos - 16384u; q < bpos; q++) t[hash64(ld64(src + q), hlog, mls)] = (u16)q;   // primed as at level 1
    const u32* const dtab = ed ? enc_dict_table(ed, mls == 6 ? EDT_MLS6 : EDT_MLS5) : nullptr;
    const u8* const dc = ed ? enc_dict_content(ed) : nullptr;
    u32 anchor = bpos; const u32 ilimit = bend - 8; u32 p0 = bpos + (bpos == 0 ? 1 : 0);
    while (p0 < ilimit) {
      const u32 step = 1 + accel + ((p0 - anchor) >> 8);
      u32 p[32], h[32], cand[32], candD[32]; bool act[32], ok[32], okD[32], rok[32]; u64 v[32];
      for (u32 l = 0; l < 32; l++) {
        p[l] = p0 + enc_probe_off(true, l, step); act[l] = p[l] < ilimit; v[l] = act[l] ? ld64(src + p[l]) : 0;
        h[l] = act[l] ? hash64(v[l], hlog, mls) : (0x80000000u | l);
      }
      for (u32 l = 0; l < 32; l++) {
        i32 low = -1; for (i32 k = (i32)l - 1; k >= 0; k--) if (h[k] == h[l]) { low = k; break; }   // __match_any_sync
        bool valid;
        if (low >= 0) { cand[l] = p[low]; valid = act[l]; } else valid = act[l] && candFrom(p[l], t[h[l] & 0xFFFFFF], cand[l]);
        ok[l] = valid && ld32(src + cand[l]) == (u32)v[l];
        okD[l] = false;
        if (ed && act[l] && !ok[l]) {
          candD[l] = dtab[hash64(v[l], ENC_DICT_HLOG, mls)];
          if (candD[l] != ENC_DICT_EMPTY) okD[l] = ld32(dc + candD[l]) == (u32)v[l];
        }
        rok[l] = act[l] && l != 0 && !(l & 1) && rep1 != 0 && rep1 <= p[l] && ld32(src + p[l] - rep1) == (u32)v[l];
      }
      i32 fl = -1, fb = -1;                                           // fb: libzstd's current0, the pair start (the fill)
      for (u32 k = 0; k < 16 && fl < 0; k++) {
        if (2 * k + 2 < 32 && rok[2 * k + 2]) { fl = 2 * k + 2; fb = 2 * k; }
        else if (ok[2 * k] || okD[2 * k]) fb = fl = 2 * k;
        else if (ok[2 * k + 1] || okD[2 * k + 1]) fb = fl = 2 * k + 1;
      }
      auto insert = [&](u32 limit) {   // ascending lanes: last writer wins; nothing at or beyond the restart position
        for (u32 l = 0; l < 32; l++) if (act[l] && p[l] < limit) t[h[l]] = (u16)p[l]; };
      if (fl < 0) { insert(0xFFFFFFFFu); p0 += 16 * step; continue; }
      u32 pos = p[fl]; const u32 kind = rok[fl] ? 0 : (ok[fl] ? 1 : 3);
      u32 cnd = kind == 0 ? pos - rep1 : (kind == 1 ? cand[fl] : candD[fl]);
      u32 off, mlen;
      if (kind == 3) {                                                 // against the dictionary content, up to its end
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
        t[hash64(ld64(src + p[fb] + 2), hlog, mls)] = (u16)(p[fb] + 2);
        t[hash64(ld64(src + p0 - 2), hlog, mls)] = (u16)(p0 - 2);
        while (rep2 != 0 && rep2 <= p0 && p0 <= ilimit && ld32(src + p0) == ld32(src + p0 - rep2)) {   // immediate repeat
          const u32 rlen = 4 + extend(p0 + 4, rep2, bend);
          std::swap(rep1, rep2);
          t[hash64(ld64(src + p0), hlog, mls)] = (u16)p0;
          seqs[2 * nseq] = ((rlen - 3) & 0xFFFF) << 16; seqs[2 * nseq + 1] = 1u | ((((rlen - 3) >> 16) & 1) << 30);
          nseq++; p0 += rlen; anchor = p0;
        }
      }
    }
    const u32 ll = bend - anchor; memcpy(lits.data() + nlits, src + anchor, ll); nlits += ll;
    st.seqs = seqs.data(); st.n = nseq; st.cap = BLOCKSIZE_MAX / 4 + 64; st.lits = lits.data(); st.nlits = nlits;
    return true;
  }
};

// raw literals section (type 0), as warp_enc_literals writes it at the negative levels; 0 = no room
u32 raw_literals(u8* out, u32 cap, const u8* lits, u32 n) {
  const u32 lh = n < 32 ? 1 : (n < 4096 ? 2 : 3);
  if (lh + n > cap) return 0;
  if (lh == 1) out[0] = (u8)(n << 3); else if (lh == 2) { u32 v = (1u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); }
  else { u32 v = (3u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); }
  for (u32 i = 0; i < n; i++) out[lh + i] = lits[i];
  return lh + n;
}

// frame assembly: dict_encoder.cpp's encode_frame_d with raw literals
u32 encode_frame_fast(const u8* src, u32 size, u8* dst, u32 cap, int level, int checksum, FastWarpMatcher& m, const EncDict* ed) {
  const u32 seqCap = BLOCKSIZE_MAX / 4 + 64;
  std::vector<u8> codes(3 * seqCap), sym(4096); std::vector<u16> ct(3 * 514 + 16);
  const u32 dictID = ed ? ed->dictID : 0;
  const u32 fhs = enc_frame_header_size(size, dictID);
  const u32 tail = checksum ? 4 : 0;
  if (cap < fhs + 3 + tail) return zerr(ZE_dstSize_tooSmall);
  u32 op = enc_frame_header(dst, size, checksum, dictID);
  u32 pos = 0, blk = 0;
  do {
    const u32 bsize = size - pos < BLOCKSIZE_MAX ? size - pos : BLOCKSIZE_MAX;
    const u32 last = pos + bsize == size;
    const u8* bstart = src + pos;
    if (op + 3 + tail > cap) return zerr(ZE_dstSize_tooSmall);
    bool rle = bsize > 0;
    for (u32 i = 1; i < bsize && rle; i++) if (bstart[i] != bstart[0]) rle = false;
    SeqStore st; st.n = 0; st.nlits = 0; st.seqs = nullptr; st.lits = nullptr; st.cap = 0;
    const bool haveSeqs = m(st, blk, bstart, bsize, rle && bsize >= 2);
    if (rle && bsize >= 2) {
      if (op + 4 + tail > cap) return zerr(ZE_dstSize_tooSmall);
      const u32 h = last | (1u << 1) | (bsize << 3);
      dst[op] = (u8)h; dst[op + 1] = (u8)(h >> 8); dst[op + 2] = (u8)(h >> 16); dst[op + 3] = bstart[0]; op += 4;
    } else {
      u32 csize = 0; bool compressed = false;
      if (haveSeqs) {
        u32 room = bsize - 1 < BLOCKSIZE_MAX - 1 ? bsize - 1 : BLOCKSIZE_MAX - 1;
        const u32 avail = cap - op - 3 - tail;
        if (room > avail) room = avail;
        u8* body = dst + op + 3;
        const EncDict* const edb = ed && ed->hasEntropy && blk == 0 ? ed : nullptr;
        const u32 l = raw_literals(body, room, st.lits, st.nlits);
        if (l) {
          const u32 s = enc_sequences_d(body + l, room - l, st, codes.data(), ct.data(), sym.data(), level, edb);
          if (s && l + s < bsize) { csize = l + s; compressed = true; }
        }
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

}  // namespace

// One frame as the compress calls write it at level -7..-1 (the checksum slot left for the caller, as k_enc_xxh fills it);
// batch_max: the largest chunk of the call (the match table's size).  use_dict: with the dictionary of hsdict_set, as the
// _using_dict calls (GENERIC when none is set, its error for a malformed one).  GENERIC for a level outside -7..-1.
extern "C" uint32_t hsfast_compress(uint8_t* dst, uint32_t cap, const uint8_t* src_in, uint32_t size, int level, int checksum,
                                    uint32_t batch_max, int use_dict) {
  if (level < -7 || level > -1) return zerr(ZE_GENERIC);
  const EncDict* ed = nullptr;
  if (use_dict) {
    if (!g_have) return zerr(ZE_GENERIC);
    ed = reinterpret_cast<const EncDict*>(g_enc.data());
    if (ed->err) return zerr(ed->err);
  }
  std::vector<u8> padded(size + 64, 0);
  u8* src = padded.data() + 16;
  if (size) memcpy(src, src_in, size);
  FastWarpMatcher m; m.src = src; m.hlog = enc_hlog_long(level, batch_max > BLOCKSIZE_MAX); m.mls = enc_mls(level);
  m.accel = (u32)-level; m.tab.assign(1u << m.hlog, 0); m.ed = ed;
  m.rep1 = ed ? ed->rep[0] : 1; m.rep2 = ed ? ed->rep[1] : 4;
  return encode_frame_fast(src, size, dst, cap, level, checksum, m, ed);
}
