// zb_blocks.cuh — block-parallel entropy decoding of multi-block frames (SURVEY.md §8f-2).
//
// A frame larger than 128 KiB is a chain of blocks.  In the reference (ZStdDecompress.cs:2033-2067) a block inherits
// exactly three things from its predecessors:
//   * the Huffman table, when its literals are "treeless"                         (litEntropy / HUFptr, :746-747)
//   * each of the LL / OF / ML tables it declares in "repeat" mode                (fseEntropy, :1062-1064)
//   * the three repeat offsets                                                    (:1576, :1596)
// The first two are defined by the HEADER of some earlier block, which any thread can parse again; only the repeat
// offsets depend on decoded data.  So every compressed block becomes a BlockUnit that the entropy kernels decode on
// their own: tables come from the defining block's header, and the repeat offsets are carried SYMBOLICALLY — an offset
// that stems from the block's (unknown) initial history is recorded as "initial entry k, decremented d times", the
// block's final history likewise; the execute stage, which walks a frame's blocks in order anyway, composes the
// histories and resolves those records as it loads them.
//
// Only structurally sound frames take this path (par_walk accepts them): every block header, literals header and
// sequence count parses, every repeat / treeless mode has a definer, the literals and records fit the frame's scratch
// regions.  Anything else stays on the frame-serial kernels, whose error handling is the reference's statement for
// statement.  Failures INSIDE a block (Huffman streams, table descriptions, the sequence bitstream) are recorded per
// unit; the execute stage meets them in block order, as the serial path does.
//
// __host__ __device__ like the rest of the stage code: tests/hostsim replays it on the CPU.
#pragma once
#include "zb_decode.cuh"

namespace zb {

enum : u32 { DEF_SELF = 0xFFFFFFFEu, DEF_DICT = 0xFFFFFFFDu, DEF_NONE = 0xFFFFFFFFu };

// frames get one unit slot per PAR_UNIT_BYTES of output capacity plus PAR_UNIT_SLACK (frames of many tiny blocks stay serial)
#define PAR_UNIT_BYTES 16384u
#define PAR_UNIT_SLACK 2u

struct BlockUnit {     // 64 bytes
  u32 frame;           // item index within the slice
  u32 body;            // offset within the item of the block's content (after its 3-byte header)
  u32 csize;           // compressed size
  u32 lit_off;         // where its Huffman literals go within the frame's literal region
  u32 rec_off;         // its header record's slot within the frame's record region
  u32 huf_def;         // frame-relative unit whose literals section carries the Huffman table in force (DEF_SELF / DEF_DICT)
  u32 tab_def[3];      // the same for the LL, OF, ML tables (indexed by KIND_*)
  // results of the entropy stages
  u32 huf_err;         // 0 or the error code of the literals
  u32 seq_err_code, seq_err_index;   // as FrameInfo::seq_err_* (index 0xFFFFFFFF = table descriptions)
  u32 rep[3];          // repeat-offset history after the block: a value, or a decrement count when symbolic
  u32 rep_sym;         // 3 bits per entry (entry i at bits 3i..3i+2): see RepSym
};
static_assert(sizeof(BlockUnit) == 64, "BlockUnit layout");

// ---- symbolic repeat offsets ------------------------------------------------------------------------------------------
// tag: 0 = v is the value; else bits 0-1 = k (1..3): the value derives from the block's initial history entry k-1,
// v counts the decrements applied to it (offset code "rep0 - 1", :1514), bit 2 = it went through the zero clamp (:1515).
// resolve() gives the value once the initial history R is known.
ZB_HD u32 repsym_resolve(u32 v, u32 tag, const u32* R) {
  if (!tag) return v;
  u32 x = R[(tag & 3) - 1];
  if (tag & 4) { x = x == 0 ? 1 : x; x = x > v ? x - v : 1; }
  return x;
}
struct RepHist {
  u32 v0, v1, v2, t0, t1, t2;
  ZB_HD void init_symbolic() { v0 = v1 = v2 = 0; t0 = 1; t1 = 2; t2 = 3; }
};
// rep_resolve (zb_decode.cuh) over (value, tag) pairs: same selection and history update; returns the offset's pair
ZB_HD void rep_resolve_sym(RepHist& h, u32 ofBits, u32 ofv, u32 llSym, u32& offV, u32& offT) {
  const bool isRep = ofBits <= 1;
  const u32 raw = (1u << (ofBits & 31)) - 3 + ofv;
  const u32 idx = ofBits + ofv + (llSym == 0);
  u32 pv = h.v0, pt = h.t0;
  if (idx == 1) { pv = h.v1; pt = h.t1; }
  if (idx == 2) { pv = h.v2; pt = h.t2; }
  const u32 dec = idx == 3 ? 1u : 0u;
  u32 cv = pv - dec; cv = cv == 0 ? 1 : cv;                             // concrete pick (zero forced to 1, as rep_resolve does)
  const u32 sv = pv + dec, stag = pt | 4;                                // symbolic pick
  const u32 kv = pt ? sv : cv, kt = pt ? stag : 0;
  offV = isRep ? kv : raw; offT = isRep ? kt : 0;
  const bool keep1 = isRep && idx == 0, keep2 = isRep && idx <= 1;
  const u32 n2v = keep2 ? h.v2 : h.v1, n2t = keep2 ? h.t2 : h.t1;
  const u32 n1v = keep1 ? h.v1 : h.v0, n1t = keep1 ? h.t1 : h.t0;
  h.v2 = n2v; h.t2 = n2t; h.v1 = n1v; h.t1 = n1t; h.v0 = offV; h.t0 = offT;
}

// Record format of a unit: as SeqRec (zb_decode.cuh) with the offset's tag in y bits 21-23 and, for a symbolic offset,
// the decrement count in z.
ZB_HD u32 rec_tag(const SeqRec& r) { return (r.y >> 21) & 7; }

// The finishing half of sequence decoding for one unit: SeqEmitter's interface, symbolic history, the unit's own
// record region (sized by the walk: header record + nbSeq slots, so it cannot overflow).
struct UnitEmitter {
  SeqRec* out; const u32* llInfo; const u32* mlInfo;
  u32 n, dpos, lpos;
  RepHist h;
  u32 err_code, err_index; bool dead;
  ZB_HD void init(SeqRec* o, const u32* lli, const u32* mli) {
    out = o; llInfo = lli; mlInfo = mli; n = 0; dpos = 0; lpos = 0; h.init_symbolic(); err_code = 0; err_index = 0; dead = false;
  }
  ZB_HD void block_begin() { n = 1; dpos = 0; lpos = 0; }
  ZB_HD void emit(u32 ofBits, u32 ofv, u32 llSym, u32 ll, u32 ml) {
    u32 ov, ot; rep_resolve_sym(h, ofBits, ofv, llSym, ov, ot);
    rec_store(out + n, dpos, lpos | ((ml >> 15) << 18) | (ot << 21), ov, ll | (ml << 17));
    n++; dpos = sat_add32(dpos, ll + ml); lpos = sat_lpos(lpos, ll);
  }
  ZB_HD void fast(u32 hi, u32 llSym, u32 mlSym, u32 ofBits, u32 mlBits, u32 llBits) {
    const u32 ofv = take_bits(hi, ofBits), mlv = take_bits(hi, mlBits), llv = take_bits(hi, llBits);
    emit(ofBits, ofv, llSym, (llInfo[llSym] & 0xFFFFFF) + llv, (mlInfo[mlSym] & 0xFFFFFF) + mlv);
  }
  ZB_HD void values(u32 ofv, u32 mlv, u32 llv, u32 llSym, u32 mlSym, u32 ofBits) {
    emit(ofBits, ofv, llSym, (llInfo[llSym] & 0xFFFFFF) + llv, (mlInfo[mlSym] & 0xFFFFFF) + mlv);
  }
  ZB_HD bool stopped() const { return dead; }
  ZB_HD void defer() {}                      // (units always run with full-size tables)
  ZB_HD void block_end(u32, u32 runnable, bool bad) {
    u32 count = n - 1;
    if (bad && runnable < count) count = runnable;
    rec_store(out, count, dpos, lpos, 0);
    if (bad) { err_code = ZE_corruption_detected; err_index = runnable; dead = true; }
  }
  ZB_HD void fail(u32, u32 code) { err_code = code; err_index = 0xFFFFFFFFu; dead = true; }
};

// ---- the structural walk ------------------------------------------------------------------------------------------------
// Walks the blocks of the data frame at body_off.  Returns the number of compressed blocks when the frame qualifies for
// the block-parallel path (>= 2 of them, every header sound, every inherited table defined, scratch regions sufficient,
// no more than maxUnits), else 0.  With units != nullptr the units are written (frame-relative definer indices).
// litCap / recCap: the frame's literal and record scratch (lit_capacity, seq_capacity of its output capacity).
ZB_HD u32 par_walk(const u8* src, u32 size, u32 body_off, u64 litCap, u64 recCap, const DictState* dict, u32 maxUnits, BlockUnit* units, u32 frame) {
  u32 pos = body_off, n = 0; u64 litRun = 0, recRun = 0;
  const u32 inherited = (dict && dict->hasEntropy) ? DEF_DICT : DEF_NONE;
  u32 lastHuf = inherited, lastTab[3] = {inherited, inherited, inherited};
  while (true) {
    BlockHdr bh;
    if (read_block_hdr(src + pos, size - pos, bh)) return 0;
    if (bh.last && n + (bh.type == 2 ? 1u : 0u) < 2) return 0;                     // single-block frames leave at their first header
    pos += 3;
    if (bh.type == 2) {
      const u8* bp = src + pos; const u32 bsz = bh.csize;
      if (bsz >= BLOCKSIZE_MAX) return 0;
      LitHdr lh; bool needs;
      if (read_lit_hdr(bp, bsz, lh, &needs)) return 0;
      if (needs && lastHuf == DEF_NONE) return 0;
      u32 nbSeq, modes, hdr;
      if (read_seq_count(bp + lh.consumed, bsz - lh.consumed, &nbSeq, &modes, &hdr)) return 0;
      if (n >= maxUnits) return 0;
      BlockUnit u;
      u.frame = frame; u.body = pos; u.csize = bsz; u.lit_off = (u32)litRun; u.rec_off = (u32)recRun;
      u.huf_def = DEF_SELF; u.tab_def[0] = u.tab_def[1] = u.tab_def[2] = DEF_SELF;
      u.huf_err = 0; u.seq_err_code = 0; u.seq_err_index = 0; u.rep[0] = u.rep[1] = u.rep[2] = 0; u.rep_sym = 1 | (2 << 3) | (3 << 6);
      if (lh.type >= 2) {
        if (litRun + lh.litSize + 3 > litCap) return 0;                            // the serial path's validate-only case
        if (lh.type == 3) u.huf_def = lastHuf; else lastHuf = n;
        litRun += lh.litSize;
      }
      if (nbSeq) {
        const int kinds[3] = {KIND_LL, KIND_OF, KIND_ML};
        const u32 modeOf[3] = {(modes >> 4) & 3, (modes >> 2) & 3, modes & 3};
        for (int k = 0; k < 3; k++) {
          if (modeOf[k] == 3) { if (lastTab[kinds[k]] == DEF_NONE) return 0; u.tab_def[kinds[k]] = lastTab[kinds[k]]; }
          else lastTab[kinds[k]] = n;
        }
        recRun += 1 + (u64)nbSeq;
        if (recRun > recCap) return 0;
      }
      if (units) units[n] = u;
      n++;
    }
    pos += bh.csize;
    if (bh.last) break;
  }
  return n >= 2 ? n : 0;
}

// ---- one unit's sequences ---------------------------------------------------------------------------------------------------
// Position of the description of table `kind` within the sequences header of the block at (bp, bsz), and its mode.
// Returns false when an earlier description of that header does not parse (the block itself then fails the same way).
template <class NormT>
ZB_HD bool unit_locate_table(const u8* bp, u32 bsz, int kind, NormT norm, const u8** desc, u32* descSize, u32* mode) {
  LitHdr lh; bool needs;
  if (read_lit_hdr(bp, bsz, lh, &needs)) return false;
  const u8* sp = bp + lh.consumed; const u32 ssz = bsz - lh.consumed;
  u32 nbSeq, modes, hdr;
  if (read_seq_count(sp, ssz, &nbSeq, &modes, &hdr) || !nbSeq) return false;
  const int kinds[3] = {KIND_LL, KIND_OF, KIND_ML};
  const u32 modeOf[3] = {(modes >> 4) & 3, (modes >> 2) & 3, modes & 3};
  for (int k = 0; k < 3; k++) {
    if (kinds[k] == kind) { *desc = sp + hdr; *descSize = ssz - hdr; *mode = modeOf[k]; return true; }
    if (modeOf[k] == 1) { if (ssz - hdr == 0) return false; hdr += 1; }
    else if (modeOf[k] == 2) {
      u32 max = kinds[k] == KIND_LL ? MaxLL : (kinds[k] == KIND_ML ? MaxML : MaxOff), tl, h;
      if (read_ncount(norm, &max, &tl, sp + hdr, ssz - hdr, &h)) return false;
      hdr += h;
    }
  }
  return false;
}

// Decodes the sequences of unit `u` (a compressed block of the item at src) into its record region `recs`.
// frameUnits: the frame's units (definer indices are relative to it).  T: the thread's table space (as seq_decode_frame).
template <class NormT, class NextT>
ZB_HD void seq_decode_unit(const u8* src, const BlockUnit& u, const BlockUnit* frameUnits, u64 window, SeqTableSet& T, UnitEmitter& em,
                           const u32* llInfo, const u32* mlInfo, NormT norm, NextT symbolNext, u32* ringMem, const DictState* dict) {
  const u8* bp = src + u.body; const u32 bsz = u.csize;
  LitHdr lh; bool needs;
  read_lit_hdr(bp, bsz, lh, &needs);                                               // sound: par_walk has parsed it
  const u8* sp = bp + lh.consumed; const u32 ssz = bsz - lh.consumed;
  u32 nbSeq, modes, hdr;
  read_seq_count(sp, ssz, &nbSeq, &modes, &hdr);
  if (!nbSeq) return;
  for (int k = 0; k < 3; k++) T.log[k] = 0;
  const int kinds[3] = {KIND_LL, KIND_OF, KIND_ML};
  const u32 modeOf[3] = {(modes >> 4) & 3, (modes >> 2) & 3, modes & 3};
  u32 e = 0;
  for (int k = 0; k < 3 && !e; k++) {                                              // the block's own descriptions, in header order
    const int kind = kinds[k]; u32 used = 0, lg = 0; bool isDef = false;
    if (modeOf[k] == 3) continue;
    e = read_seq_table(modeOf[k], kind, sp + hdr, ssz - hdr, T.space[kind], T.stride, &lg, &isDef, true, &used, norm, symbolNext);
    if (!e) { hdr += used; T.log[kind] = lg; if (isDef) seq_use_default(T, kind); }
  }
  for (int k = 0; k < 3 && !e; k++) {                                              // inherited tables: rebuilt from their definer
    const int kind = kinds[k];
    if (modeOf[k] != 3) continue;
    const u32 def = u.tab_def[kind];
    if (def == DEF_DICT) {
      const u32 cells = 1u << dict->log[kind];
      for (u32 c = 0; c < cells; c++) T.space[kind][c * T.stride] = dict->cells[kind][c];
      T.log[kind] = dict->log[kind];
    } else {
      const BlockUnit& d = frameUnits[def];
      const u8* desc; u32 descSize, mode, used = 0, lg = 0; bool isDef = false;
      if (!unit_locate_table(src + d.body, d.csize, kind, norm, &desc, &descSize, &mode)) { e = ZE_corruption_detected; break; }
      e = read_seq_table(mode, kind, desc, descSize, T.space[kind], T.stride, &lg, &isDef, true, &used, norm, symbolNext);
      if (!e) { T.log[kind] = lg; if (isDef) seq_use_default(T, kind); }
    }
  }
  if (e) { em.fail(0, ZE_corruption_detected); return; }
  seq_decode_bitstream(sp + hdr, ssz - hdr, nbSeq, window, T, em, llInfo, mlInfo, ringMem, 0);
}

}  // namespace zb
