// zb_decode.cuh — per-thread bodies of the entropy stages of the GPU decoder.
//
//   seq_decode_frame : one thread walks one frame's blocks, builds the LL/OF/ML tables in (bank-interleaved)
//                      shared memory and hands every sequence of the bitstreams to a sink; SeqEmitter turns them into
//                      16-byte records in HBM scratch.
//   huf_*            : one thread per Huffman stream (4 per frame) decodes literals into HBM scratch from a
//                      shared-memory decode table built by the frame's first lane.
//
// They are __host__ __device__ so that tests/hostsim can replay exactly this code on the CPU.
#pragma once
#include "zb_format.cuh"

namespace zb {

// 16-byte sequence record consumed by the execute stage.  A record is self-describing — it carries where its
// bytes go and where its literals come from — so the execute stage needs no prefix sums and its warps can work on
// different groups of a block's records without a positional chain between them.
//   x = dpos : output position of the sequence's literal run, relative to the block's first output byte
//              (saturates at 0xFFFFFFFF: such a record can never pass the capacity check)
//   y = lpos (18 bits: position of its literals within the block's literals, saturates at 0x3FFFF)
//       | matchLength >> 15 << 18 (3 bits: matchLength <= 131074)
//   z = offset (>= 1 for a well-formed match; garbage offsets of corrupted streams use all 32 bits)
//   w = litLength (17 bits) | (matchLength & 0x7FFF) << 17
// The records of one compressed block are preceded by one header record:
//   x = number of records that follow, y = output bytes of those records (saturating), z = literal bytes they take
//   (saturating at 0x3FFFF), w = 0
struct alignas(16) SeqRec { u32 x, y, z, w; };
ZB_HD void rec_store(SeqRec* p, u32 x, u32 y, u32 z, u32 w) {
#if defined(__CUDA_ARCH__)
  *reinterpret_cast<uint4*>(p) = make_uint4(x, y, z, w);
#else
  p->x = x; p->y = y; p->z = z; p->w = w;
#endif
}
ZB_HD u32 rec_ll(const SeqRec& r) { return r.w & 0x1FFFF; }
ZB_HD u32 rec_ml(const SeqRec& r) { return (r.w >> 17) | (((r.y >> 18) & 7) << 15); }
ZB_HD u32 rec_lpos(const SeqRec& r) { return r.y & 0x3FFFF; }
ZB_HD u32 sat_add32(u32 a, u32 b) { const u32 s = a + b; return s < a ? 0xFFFFFFFFu : s; }
ZB_HD u32 sat_lpos(u32 lpos, u32 ll) { const u32 s = lpos + ll; return s > 0x3FFFFu ? 0x3FFFFu : s; }

// Capacity rule shared with the host side: records for a frame whose output capacity is `cap` bytes.
// Every sequence yields >= 3 bytes and each block with sequences adds one header record, so a frame that fits
// its capacity needs fewer than 2*(cap/3) + 24 records; running out of room therefore means dstSize_tooSmall.
ZB_HD u64 seq_capacity(u64 cap) { return 2 * (cap / 3) + 24; }

struct SeqTableSet {
  u32 cap[3] = {9, 9, 9};   // table log each space can hold (KIND_LL, KIND_OF, KIND_ML); smaller in the kernels for frames of few sequences
  u16* space[3];            // lane-private cells for LL, OF, ML (index with *stride): the tables in force
  u32 stride;
  const u16* defs[3];       // predefined tables, stride 1: a block that selects one gets a copy in its space (seq_use_default)
  u32 log[3];
};
// Every table the sequence loop reads sits in the lane's space, so that a cell's address is the state times one stride
// (a shift on the device) whichever mode a block chose.  The predefined logs (6 / 5 / 6) fit every class's space.
ZB_HD void seq_use_default(SeqTableSet& T, int kind) {
  for (u32 u = 0; u < (1u << T.log[kind]); u++) T.space[kind][u * T.stride] = T.defs[kind][u];
}

struct SeqFrameOut {
  u32 err_block, err_code, err_index;
};

// n bits (0..32) from the top of a left-aligned 64-bit window; the double shift makes n == 0 yield 0
// (the reference's LookBits does the same, BitStream.cs:412-416)
ZB_HD u32 top_bits(u64 w, u32 n) { return (u32)((w >> 1) >> (63 - n)); }

// Offset value of one sequence and the repeat-offset history update (DecodeSequence :1487-1531), written
// without data-dependent branches.  ofBits is the offset code, ofv its extra bits, llSym the literal-length code.
ZB_HD u32 rep_resolve(u32& rep0, u32& rep1, u32& rep2, u32 ofBits, u32 ofv, u32 llSym) {
  const bool isRep = ofBits <= 1;
  const u32 raw = (1u << (ofBits & 31)) - 3 + ofv;                     // OF_base + extra bits for codes >= 2 (:1088-1092)
  const u32 idx = ofBits + ofv + (llSym == 0);                         // codes 0/1: repeat-offset index 0..3 (base 0 / 1, ofv = 0 for code 0)
  u32 pick = rep0;
  pick = idx == 1 ? rep1 : pick;
  pick = idx == 2 ? rep2 : pick;
  pick = idx == 3 ? rep0 - 1 : pick;
  pick = pick == 0 ? 1 : pick;                                         // 0 is not valid: forced to 1 (:1515)
  const u32 offset = isRep ? pick : raw;
  const bool keep1 = isRep && idx == 0;                                // history is untouched only when idx == 0
  const bool keep2 = isRep && idx <= 1;
  const u32 n2 = keep2 ? rep2 : rep1, n1 = keep1 ? rep1 : rep0;
  rep2 = n2; rep1 = n1; rep0 = offset;
  return offset;
}

// ---------------------------------------------------------------------------------------------------
// Over-read emulation.  The reference reads its backward bitstream through a 4-byte container
// (BitStream.cs:322-489, size_t = UInt32).  A sequence whose value bits reach below the stream start is not
// rejected on the spot: the reads return whatever the container shifts produce (shift counts are taken mod 32),
// the sequence is executed, and only the next loop test (:1582) sees the overflow — never, if it was the block's
// last sequence.  To give the same verdicts and bytes, the careful loop recomputes such a sequence's values with
// the container arithmetic below.  The container state at a sequence's start follows from the unread-bit count P
// alone, because the loop test has just reloaded: bitsConsumed is normalised to < 8 unless the container already
// sits on the stream's first bytes.
// ---------------------------------------------------------------------------------------------------
struct RefBits {
  const u8* s; u32 n;   // the stream
  i32 k;                // container = bytes [k, k+4) of the stream
  u32 bc, C;            // bitsConsumed, bitContainer
};
ZB_HD void refbits_load(RefBits& b) {
  if (b.n >= 4) { b.C = ld32(b.s + b.k); return; }
  b.C = b.s[0]; if (b.n >= 2) b.C |= (u32)b.s[1] << 8; if (b.n >= 3) b.C |= (u32)b.s[2] << 16;       // BitStream.cs:343-367
}
ZB_HD void refbits_at(RefBits& b, const u8* s, u32 n, i32 P) {                  // state right after a reload, P >= 0
  b.s = s; b.n = n;
  const i32 bcn = (8 - (P & 7)) & 7, above = P - 32 + bcn;                        // bits above a normalised container
  if (n >= 4 && above >= 0) { b.k = above >> 3; b.bc = (u32)bcn; } else { b.k = 0; b.bc = (u32)(32 - P); }
  refbits_load(b);
}
ZB_HD u32 refbits_read_fast(RefBits& b, u32 nb) { u32 v = (b.C << (b.bc & 31)) >> ((32 - nb) & 31); b.bc += nb; return v; }   // :445-451
ZB_HD void refbits_reload(RefBits& b) {                                          // BitStream.cs:458-489
  if (b.bc > 32 || b.k == 0) return;
  u32 nb = b.bc >> 3;
  if (b.k >= 4 || (i32)nb <= b.k) { b.k -= (i32)nb; b.bc -= nb * 8; } else { b.bc -= (u32)b.k * 8; b.k = 0; }
  refbits_load(b);
}
// value bits of one sequence in the reference's read order and reload schedule (DecodeSequence :1487-1545, MEM_32bits)
// longVariant: the block runs DecodeSequenceLong (:1620-1706), which splits an offset at a fixed 24 bits (:1642-1647)
ZB_HD void seq_values_ref32(const u8* s, u32 n, i32 P, bool longOffsets, bool longVariant, u32 ofBits, u32 mlBits, u32 llBits, u32& ofv, u32& mlv, u32& llv) {
  RefBits b; refbits_at(b, s, n, P);
  ofv = 0;
  if (ofBits) {
    if (longOffsets && (longVariant || ofBits >= 25)) {                            // :1494-1501
      const u32 room = longVariant ? 24 : 32 - b.bc, extra = ofBits - (ofBits < room ? ofBits : room);
      ofv = refbits_read_fast(b, ofBits - extra) << (extra & 31);
      refbits_reload(b);
      if (extra) ofv += refbits_read_fast(b, extra);
    } else { ofv = refbits_read_fast(b, ofBits); refbits_reload(b); }              // :1504-1506
  }
  mlv = mlBits ? refbits_read_fast(b, mlBits) : 0;                                 // :1534
  if (mlBits + llBits >= 20) refbits_reload(b);                                    // :1536 (25 - 5)
  llv = llBits ? refbits_read_fast(b, llBits) : 0;                                 // :1542
}

// ---------------------------------------------------------------------------------------------------
// Sequence decoding is split in two halves that meet at a narrow interface (a "sink"):
//   the CHAIN half (seq_decode_frame) owns what is serially dependent from one sequence to the next — the three FSE
//   states and the bit cursor (DecodeSequence :1473-1553 without its value arithmetic) — and hands every sequence
//   over as (32 stream bits that begin with its value bits, the three symbols);
//   the FINISHING half (SeqEmitter) extracts the value bits, applies the repeat-offset rules (:1509-1530), keeps the
//   running output / literal positions and writes the records.
// The kernel (k_seq) and the CPU replay (tests/hostsim) plug the emitter in directly.  (Measured in round 2: the halves
// on two warps of one CTA with a per-lane shared-memory queue between them — see k_seq in decode_kernels.cu; slower.)
// ---------------------------------------------------------------------------------------------------
struct SeqEmitter {
  SeqRec* out; u32 cap; const u32* llInfo; const u32* mlInfo;
  u32 n;                          // record slots used so far (headers included)
  u32 hdrSlot, dpos, lpos;        // the current block: its header slot, running output / literal positions
  u32 rep0, rep1, rep2;           // ZStdInternal.cs:111, ZStdDecompress.cs:2492
  bool dead;                      // the frame's first entropy-level error has been recorded: later blocks are ignored
  bool deferred;                  // a table did not fit this instantiation's space: nothing of this attempt counts
  SeqFrameOut res;
  ZB_HD void init(SeqRec* o, u64 cap64, const u32* lli, const u32* mli) {
    out = o; cap = (u32)cap64; llInfo = lli; mlInfo = mli;        // seq_capacity of a u32 capacity fits 32 bits
    n = 0; hdrSlot = 0; dpos = 0; lpos = 0; rep0 = 1; rep1 = 4; rep2 = 8; dead = false; deferred = false;
    res.err_block = 0xFFFFFFFFu; res.err_code = 0; res.err_index = 0;
  }
  ZB_HD void set_reps(const u32* r) { rep0 = r[0]; rep1 = r[1]; rep2 = r[2]; }          // a dictionary's repeat offsets (:2436-2442)
  ZB_HD void block_begin() { if (dead) return; hdrSlot = n++; dpos = 0; lpos = 0; }   // the block's header record is written last
  ZB_HD void emit(u32 ofBits, u32 ofv, u32 llSym, u32 ll, u32 ml) {
    const u32 offset = rep_resolve(rep0, rep1, rep2, ofBits, ofv, llSym);
    if (n < cap) rec_store(out + n, dpos, lpos | ((ml >> 15) << 18), offset, ll | (ml << 17));
    n++; dpos = sat_add32(dpos, ll + ml); lpos = sat_lpos(lpos, ll);
  }
  // a sequence of the fast path: hi = 32 stream bits whose top bits are its value bits (fewer than 32 of them), in the
  // reference's read order offset, matchLength, litLength (:1504, :1534, :1542)
  ZB_HD void fast(u32 hi, u32 llSym, u32 mlSym, u32 ofBits, u32 mlBits, u32 llBits) {
    const u32 ofv = take_bits(hi, ofBits), mlv = take_bits(hi, mlBits), llv = take_bits(hi, llBits);
    emit(ofBits, ofv, llSym, (llInfo[llSym] & 0xFFFFFF) + llv, (mlInfo[mlSym] & 0xFFFFFF) + mlv);
  }
  // a sequence whose value bits the chain half had to extract itself (stream tail, >= 32 value bits, over-reads)
  ZB_HD void values(u32 ofv, u32 mlv, u32 llv, u32 llSym, u32 mlSym, u32 ofBits) {
    emit(ofBits, ofv, llSym, (llInfo[llSym] & 0xFFFFFF) + llv, (mlInfo[mlSym] & 0xFFFFFF) + mlv);
  }
  // true once the frame's first entropy-level error is recorded: the chain half stops (nothing it decodes is used)
  ZB_HD bool stopped() const { return dead; }
  ZB_HD void defer() { deferred = true; }
  // bad = the bitstream failed (:1577, :1582 -> corruption_detected); runnable = how many of the block's sequences the
  // reference has executed by then (all that were decoded in the regular loop, four fewer in the look-ahead loop)
  ZB_HD void block_end(u32 blk, u32 runnable, bool bad) {
    if (dead) return;
    // header record: how many records the execute stage may run (those that fit the region)
    const bool overflow = n > cap;
    u32 count = (overflow ? cap : n) - hdrSlot - 1;
    if (bad && runnable < count) count = runnable;
    if (hdrSlot < cap) rec_store(out + hdrSlot, count, dpos, lpos, 0);
    if (overflow) { res.err_block = blk; res.err_code = ZE_dstSize_tooSmall; res.err_index = 0; dead = true; }
    else if (bad) { res.err_block = blk; res.err_code = ZE_corruption_detected; res.err_index = runnable; dead = true; }
  }
  // the block failed before its first sequence (count / table headers)
  ZB_HD void fail(u32 blk, u32 code) { if (dead) return; res.err_block = blk; res.err_code = code; res.err_index = 0xFFFFFFFFu; dead = true; }
};

// The bitstream of one compressed block: nbSeq sequences out of bits[0..nbytes) with the tables in force (T.space, T.log)
// go to `sink` (block_begin ... block_end).  Returns true when the frame cannot go on (the stream failed or the sink has
// stopped).  blk = the block's index for the sink's error record.
template <class Sink>
ZB_HD bool seq_decode_bitstream(const u8* bits, u32 nbytes, u32 nbSeq, u64 window, const SeqTableSet& T, Sink& sink,
                                const u32* llInfo, const u32* mlInfo, u32* ringMem, u32 blk) {
  // Windows above 16 MiB whose offset table has >= 20/256 cells of more than 22 extra bits run the sequence loop
  // that decodes four sequences ahead of their execution (:1898-1905, GetLongOffsetsShare :1845-1865)
  bool longVariant = false;
  if (window > (1u << 24)) {
    const u32 lg = T.log[KIND_OF]; u32 total = 0;
    for (u32 u = 0; u < (1u << lg); u++) total += (T.space[KIND_OF][u * T.stride] >> 10) > 22;
    longVariant = (total << (8 - lg)) >= 20;
  }
  // ---- bitstream ----
  BitCursor c;
  sink.block_begin();
  u32 decoded = 0; bool bad = false;
  if (!bc_init(c, bits, nbytes)) bad = true;                          // :1577 -> corruption_detected
  if (!bad) {
    i32 P = c.P;
    const u16 *tLL = T.space[KIND_LL], *tOF = T.space[KIND_OF], *tML = T.space[KIND_ML];
    const u32 S = T.stride;
    u32 stLL, stOF, stML;
    { u64 w = bc_window64(c, P); u32 lg = T.log[KIND_LL]; stLL = top_bits(w, lg); w <<= lg; P -= (i32)lg;
      lg = T.log[KIND_OF]; stOF = top_bits(w, lg); w <<= lg; P -= (i32)lg;
      lg = T.log[KIND_ML]; stML = top_bits(w, lg); P -= (i32)lg; }             // :1578-1580 (<= 26 bits)
    u32 i = 0;
    // ---- fast loop: >= 128 unread bits, so no over-read is possible (a sequence takes <= 89 bits); leaves to
    //      the careful loop when a sequence carries >= 32 value bits (rare: very long lengths / offsets).
    //      The next states and cursor are computed ahead of that test, so that their dependent chain (cell -> extra-bit
    //      counts -> state bits -> next cell) does not wait behind it; the sink then gets the sequence ----
    BitRing ring;
    if (nbSeq && P >= 128) ring_init(ring, ringMem, bits, nbytes);
    while (i < nbSeq && P >= 128) {
      u32 lo, hi;
      ring_window(ring, P, lo, hi);                                          // 64-bit window ending at P
      const u32 yLL = tLL[stLL * S], yOF = tOF[stOF * S], yML = tML[stML * S];
      const u32 llSym = yLL >> 10, mlSym = yML >> 10, ofBits = yOF >> 10;   // the offset code is its own extra-bit count
      const u32 llBits = llInfo[llSym] >> 24, mlBits = mlInfo[mlSym] >> 24;
      const u32 valBits = ofBits + mlBits + llBits;
      // state update LL, ML, OF (:1547-1550) from the 32 bits after the value bits; w * 2^n drops n of them
      const u32 uLL = cell_unit(yLL), uML = cell_unit(yML), uOF = cell_unit(yOF), uLM = uLL * uML;
      const u32 h2 = fshl(lo, hi, valBits);
      const u32 nLL = cell_next(yLL, uLL, h2), nML = cell_next(yML, uML, h2 * uLL), nOF = cell_next(yOF, uOF, h2 * uLM);
      const i32 Pn = P - (i32)(valBits + highbit(uLM * uOF));                // the units multiply to 2^(state bits)
      // the one rare exit of the loop: >= 32 value bits (they do not fit the word handed over) — nothing has been
      // committed yet, the careful loop redoes this sequence
      if (valBits >= 32) break;
      sink.fast(hi, llSym, mlSym, ofBits, mlBits, llBits);
      stLL = nLL; stML = nML; stOF = nOF;
      ring_advance(ring, Pn);
      P = Pn; i++;
    }
    decoded = i;
    // ---- careful loop: stream tail and oversized sequences ----
    for (; i < nbSeq; i++) {
      if (P < 0) { bad = true; break; }                                      // loop test :1582 (overflow)
      const u64 w0 = bc_window64(c, P);
      const u32 yLL = tLL[stLL * S], yOF = tOF[stOF * S], yML = tML[stML * S];
      const u32 llSym = yLL >> 10, mlSym = yML >> 10, ofBits = yOF >> 10;
      const u32 llBits = llInfo[llSym] >> 24, mlBits = mlInfo[mlSym] >> 24;
      const u32 lLL = yLL & 0x3FF, lOF = yOF & 0x3FF, lML = yML & 0x3FF;
      const u32 nLL = cell_nb(lLL), nML = cell_nb(lML), nOF = cell_nb(lOF);
      const u32 valBits = ofBits + mlBits + llBits, stBits = nLL + nML + nOF;
      u64 w = w0;
      u32 ofv = top_bits(w, ofBits); w <<= ofBits;
      u32 mlv = top_bits(w, mlBits); w <<= mlBits;
      u32 llv = top_bits(w, llBits); w <<= llBits;
      const i32 Pv = P - (i32)valBits;
      if (Pv < 0) seq_values_ref32(bits, nbytes, P, window > (1ull << 25), longVariant, ofBits, mlBits, llBits, ofv, mlv, llv);   // over-read: the reference's container garbage
      else if (valBits + stBits > 64) w = bc_window64(c, Pv);                // rare: more than 64 bits in one sequence
      sink.values(ofv, mlv, llv, llSym, mlSym, ofBits);
      decoded++;
      // past the last sequence these bits do not exist (the stream ends after its value bits)
      stLL = cell_base(lLL) + top_bits(w, nLL); w <<= nLL;
      stML = cell_base(lML) + top_bits(w, nML); w <<= nML;
      stOF = cell_base(lOF) + top_bits(w, nOF);
      P = Pv - (i32)stBits;
    }
  }
  // the look-ahead loop has executed all but the last four sequences when the stream runs out (:1748-1764)
  if (bad && longVariant) decoded = decoded > 4 ? decoded - 4 : 0;
  sink.block_end(blk, decoded, bad);
  return bad || sink.stopped();
}

// Walks the frame at item `src` (size bytes, first block header at body_off) and decodes every compressed
// block's sequences into `sink` (block_begin / fast / values / block_end / fail / stopped, see SeqEmitter).  Stops silently at
// structural errors that the execute stage will report itself from the same headers.
// llInfo/mlInfo: per-symbol base | extra bits << 24 (ll_info/ml_info); norm/symbolNext: >= 53 entries of per-thread scratch each;
// ringMem: ZB_RING_WORDS words of per-thread bitstream read-ahead (BitRing), 16-byte aligned.
// dict: the context's dictionary (may be null): its sequence tables are what repeat mode refers to until a block
// brings its own (fseEntropy = 1 after ZSTD_decompress_insertDictionary, :2468).
template <class Sink, class NormT, class NextT>
ZB_HD void seq_decode_frame(const u8* src, u32 size, u32 body_off, u64 window, SeqTableSet& T, Sink& sink,
                            const u32* llInfo, const u32* mlInfo, NormT norm, NextT symbolNext, u32* ringMem, const DictState* dict = nullptr) {
  u32 pos = body_off, blk = 0;
  bool haveRepeat = false;
  for (int k = 0; k < 3; k++) T.log[k] = 0;
  if (dict && dict->hasEntropy) {
    for (int k = 0; k < 3; k++) {
      const u32 n = 1u << dict->log[k];
      for (u32 u = 0; u < n; u++) T.space[k][u * T.stride] = dict->cells[k][u];
      T.log[k] = dict->log[k];
    }
    haveRepeat = true;
  }
  while (true) {
    BlockHdr bh;
    if (read_block_hdr(src + pos, size - pos, bh)) return;
    pos += 3;
    if (bh.type == 2) {
      const u8* bp = src + pos; u32 bsz = bh.csize;
      if (bsz >= BLOCKSIZE_MAX) return;                                            // :1880
      LitHdr lh; bool needs;
      if (read_lit_hdr(bp, bsz, lh, &needs)) return;
      const u8* sp = bp + lh.consumed; u32 ssz = bsz - lh.consumed;
      u32 nbSeq, modes, hdr;
      u32 e = read_seq_count(sp, ssz, &nbSeq, &modes, &hdr);
      if (e) { sink.fail(blk, e); return; }
      if (nbSeq) {
        // tables in the reference's order LL, OF, ML (:1149-1176); any failure is corruption_detected
        const int kinds[3] = {KIND_LL, KIND_OF, KIND_ML};
        const u32 modeOf[3] = {(modes >> 4) & 3, (modes >> 2) & 3, modes & 3};
        for (int k = 0; k < 3 && !e; k++) {
          int kind = kinds[k]; u32 used, lg = T.log[kind]; bool isDef = false;
          u32 m = modeOf[k];
          e = read_seq_table(m, kind, sp + hdr, ssz - hdr, T.space[kind], T.stride, &lg, &isDef, haveRepeat, &used, norm, symbolNext, T.cap[kind]);
          if (e == ZB_TABLE_TOO_LARGE) { sink.defer(); return; }                   // this frame belongs to the instantiation with full-size tables
          if (!e) {
            hdr += used;
            if (m != 3) {
              T.log[kind] = lg;
              if (isDef) seq_use_default(T, kind);
            }
          }
        }
        if (e) { sink.fail(blk, ZE_corruption_detected); return; }
        haveRepeat = true;                                                         // fseEntropy = 1 (:1575)
        if (seq_decode_bitstream(sp + hdr, ssz - hdr, nbSeq, window, T, sink, llInfo, mlInfo, ringMem, blk)) return;
      }
    }
    pos += bh.csize; blk++;
    if (bh.last) return;
  }
}

// ---------------------------------------------------------------------------------------------------
// Huffman literals
// ---------------------------------------------------------------------------------------------------
// Stream layout of a literals section body (after the optional weight header), HufDecompress.cs:266-307:
// 4 streams: 6-byte jump table then the streams; stream k (k<3) regenerates seg=(n+3)/4 bytes at out+k*seg,
// the 4th regenerates max(0, n-3*seg) at out+3*seg.  1 stream: the whole body regenerates n bytes.
struct HufStream { const u8* src; u32 len; u32 outOfs; u32 count; };

// Returns false when the jump table is inconsistent (corruption_detected in the reference).
ZB_HD bool huf_split4(const u8* body, u32 bodySize, u32 n, u32 lane, HufStream& s) {
  if (bodySize < 10) return false;                                                 // :269
  u32 l1 = ld16(body), l2 = ld16(body + 2), l3 = ld16(body + 4);
  u32 l4 = bodySize - (l1 + l2 + l3 + 6);
  if (l4 > bodySize) return false;                                                 // :303
  u32 seg = (n + 3) / 4;
  u32 start = 6, len = l1;
  if (lane == 1) { start = 6 + l1; len = l2; } else if (lane == 2) { start = 6 + l1 + l2; len = l3; } else if (lane == 3) { start = 6 + l1 + l2 + l3; len = l4; }
  s.src = body + start; s.len = len; s.outOfs = lane * seg;
  s.count = lane < 3 ? seg : (n > 3 * seg ? n - 3 * seg : 0);
  return true;
}

// One symbol: the cell for the stream bits at the top of the left-aligned window w.  T.root = 2^T.rootLog cells
// (huf_fill_root), T.full / T.side = the full table for the codes the root does not hold (huf_fill_table: 2^T.log cells,
// log 12 folded with its side table).
struct HufTabs { const u16* root; u32 rootLog; const u16* full; const u8* side; u32 log; };
// LONGS = false: the table log does not exceed the root log, no root cell is HUF_LONG — the test stays out of the chain
// of dependent lookups that bounds the decoder
template <bool LONGS>
ZB_HD u32 huf_cell(const HufTabs& T, u64 w) {
  u32 c = T.root[(u32)(w >> (64 - T.rootLog))];
  if (LONGS && c >= HUF_LONG) {
    if (T.log > HUF_TABLE_LOG) { const u32 i12 = (u32)(w >> 52), cell = T.full[i12 >> 1]; c = (cell >> 8) == 12 ? (12u << 8) | T.side[i12] : cell; }
    else c = T.full[(u32)(w >> (64 - T.log))];
  }
  return c;
}
template <bool LONGS>
ZB_HD u32 huf_cell32(const HufTabs& T, u32 w32) {
  u32 c = T.root[w32 >> (32 - T.rootLog)];
  if (LONGS && c >= HUF_LONG) c = huf_cell<true>(T, (u64)w32 << 32);
  return c;
}

// Decodes `count` symbols of one backward stream into out[0..count).  true iff the stream was consumed
// exactly (EndOfDStream, HufDecompress.cs:350-353 / :261) — which also implies it was never over-read.
template <bool LONGS>
ZB_HD bool huf_decode_stream_t(const u8* src, u32 len, u8* out, u32 count, const HufTabs& T, u32* ringMem) {
  BitCursor c;
  if (!bc_init(c, src, len)) return false;                                         // InitDStream errors :304-307
  i32 P = c.P;
  u32 left = count;
  // head: reach 4-byte alignment of the output
  while (left && ((uintptr_t)out & 3)) {
    const u32 cell = huf_cell<LONGS>(T, bc_window64(c, P));
    *out++ = (u8)cell; P -= (i32)(cell >> 8); left--;
  }
  // fast loop: 4 symbols (<= 48 bits) per iteration out of the shared-memory ring
  if (left >= 4 && P >= 128) {
    BitRing ring;
    ring_init(ring, ringMem, src, len);
    while (left >= 4 && P >= 128) {
      u32 lo, hi;
      ring_window(ring, P, lo, hi);
      const u32 c0 = huf_cell32<LONGS>(T, hi); u32 used = c0 >> 8;
      const u32 c1 = huf_cell32<LONGS>(T, fshl(lo, hi, used)); used += c1 >> 8;
      const u32 c2 = huf_cell32<LONGS>(T, fshl(lo, hi, used)); used += c2 >> 8;
      const u32 c3 = huf_cell32<LONGS>(T, used < 32 ? fshl(lo, hi, used) : (lo << (used - 32))); used += c3 >> 8;
      *(u32*)out = (c0 & 0xFF) | ((c1 & 0xFF) << 8) | ((c2 & 0xFF) << 16) | ((c3 & 0xFF) << 24);
      out += 4; left -= 4;
      P -= (i32)used;
      ring_advance(ring, P);
    }
  }
  while (left >= 4) {
    u64 w = bc_window64(c, P);
    const u32 c0 = huf_cell<LONGS>(T, w); w <<= (c0 >> 8);
    const u32 c1 = huf_cell<LONGS>(T, w); w <<= (c1 >> 8);
    const u32 c2 = huf_cell<LONGS>(T, w); w <<= (c2 >> 8);
    const u32 c3 = huf_cell<LONGS>(T, w);
    P -= (i32)((c0 >> 8) + (c1 >> 8) + (c2 >> 8) + (c3 >> 8));
    *(u32*)out = (c0 & 0xFF) | ((c1 & 0xFF) << 8) | ((c2 & 0xFF) << 16) | ((c3 & 0xFF) << 24);
    out += 4; left -= 4;
  }
  while (left) {
    const u32 cell = huf_cell<LONGS>(T, bc_window64(c, P));
    *out++ = (u8)cell; P -= (i32)(cell >> 8); left--;
  }
  return P == 0;
}
ZB_HD bool huf_decode_stream(const u8* src, u32 len, u8* out, u32 count, const HufTabs& T, u32* ringMem) {
  return T.log > T.rootLog ? huf_decode_stream_t<true>(src, len, out, count, T, ringMem) : huf_decode_stream_t<false>(src, len, out, count, T, ringMem);
}

// Validation without output: same verdict as huf_decode_stream.  Used when a block's literals cannot fit the
// frame's literal scratch — the frame is then certain to fail, but whether with corruption_detected (here) or with
// the execute stage's dstSize_tooSmall depends on whether the streams are well formed (HufDecompress.cs:350-353).
ZB_HD bool huf_check_stream(const u8* src, u32 len, u32 count, const HufTabs& T) {
  BitCursor c;
  if (!bc_init(c, src, len)) return false;
  i32 P = c.P;
  for (u32 left = count; left; left--) {
    if (P < 0) return false;
    P -= (i32)(huf_cell<true>(T, bc_window64(c, P)) >> 8);
  }
  return P == 0;
}

}  // namespace zb
