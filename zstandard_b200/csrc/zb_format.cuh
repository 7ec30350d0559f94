// zb_format.cuh — zstd frame / block / entropy-header parsing for the GPU decoder.
//
// Each function states the reference code whose behaviour (accept/reject set, error code, decoded value) it
// must reproduce; paths are relative to /root/reference/csharp/src/.  The code is written for one GPU thread
// per frame (or per Huffman stream): plain scalar control flow over bytes in global memory, tables in shared
// memory addressed through (pointer, stride) so that per-lane tables can be bank-interleaved.
#pragma once
#include "zb_common.cuh"

namespace zb {

// =====================================================================================================
// Item / frame header  (ZStdDecompress.cs:2096-2160 multi-frame loop head, :2008-2030, :389-499, :628-637)
// =====================================================================================================
// Outcome: returns true when a data frame was found and its header is valid (fi filled, later stages run);
// returns false when the item's result is already final (*result set).
// start / out_base: where in the item to look and how many bytes its earlier data frames produced (0, 0 on the
// first pass; the execute stage's next_off and running total on later passes of a multi-frame item).
// dictErr / ctxDictID: state of the context's dictionary (ZSTD_decompressBegin_usingDict :2501-2507 runs before every
// data frame and fails it with dictionary_corrupted; DecodeFrameHeader :633 compares the frame's dictionary id).
ZB_HD bool parse_item(const u8* src, u32 size, FrameInfo& fi, u32* result, u32 start = 0, u32 out_base = 0, u32 dictErr = 0, u32 ctxDictID = 0) {
  fi.flags = 0; fi.body_off = 0; fi.fcs = 0; fi.window = 0;
  fi.huf_err_block = 0xFFFFFFFFu; fi.huf_err_code = 0; fi.seq_err_block = 0xFFFFFFFFu; fi.seq_err_code = 0; fi.seq_err_index = 0;
  fi.trailer_off = 0; fi.decoded = 0; fi.out_base = out_base; fi.next_off = 0; fi.unit_base = 0; fi.unit_count = 0;
  u32 pos = start;
  while (true) {
    u32 rem = size - pos;
    if (rem < 5) { *result = rem ? zerr(ZE_srcSize_wrong) : out_base; fi.flags = FI_DONE; return false; }   // :2111, :2156
    u32 magic = ld32(src + pos);
    if (magic == MAGIC) break;
    if ((magic & 0xFFFFFFF0u) != MAGIC_SKIP) { *result = zerr(ZE_prefix_unknown); fi.flags = FI_DONE; return false; }
    if (rem < 8) { *result = zerr(ZE_srcSize_wrong); fi.flags = FI_DONE; return false; }
    u32 skip = ld32(src + pos + 4) + 8u;   // 32-bit wrap, as the reference's size_t = UInt32
    if (rem < skip) { *result = zerr(ZE_srcSize_wrong); fi.flags = FI_DONE; return false; }
    pos += skip;
  }
  if (dictErr) { *result = zerr(dictErr); fi.flags = FI_DONE; return false; }
  const u8* ip = src + pos; u32 rem = size - pos;
  u32 e = 0;
  if (rem < 6 + 3) e = ZE_srcSize_wrong;                                           // :2019
  u32 fhd = 0, fhs = 0;
  if (!e) {
    fhd = ip[4];
    u32 did = fhd & 3, single = (fhd >> 5) & 1, fcsId = fhd >> 6;
    fhs = 5 + (single ? 0 : 1) + (did == 3 ? 4 : did) + (fcsId == 0 ? 0 : (1u << fcsId)) + ((single && fcsId == 0) ? 1 : 0);   // :389-403
    if (rem < fhs + 3) e = ZE_srcSize_wrong;                                       // :2026
  }
  if (!e && (fhd & 0x08)) e = ZE_frameParameter_unsupported;                       // :461
  if (!e) {
    u32 p = 5, did = fhd & 3, single = (fhd >> 5) & 1, fcsId = fhd >> 6;
    u64 window = 0, fcs = 0; bool known = false; u32 dictID = 0;
    if (!single) {
      u32 wl = ip[p++], wlog = (wl >> 3) + 10;
      if (wlog > 30) e = ZE_frameParameter_windowTooLarge;                         // :468
      window = 1ull << wlog; window += (window >> 3) * (wl & 7);
    }
    if (!e) {
      if (did == 1) { dictID = ip[p]; p += 1; } else if (did == 2) { dictID = ld16(ip + p); p += 2; } else if (did == 3) { dictID = ld32(ip + p); p += 4; }
      if (fcsId == 0) { if (single) { fcs = ip[p]; known = true; } }
      else if (fcsId == 1) { fcs = ld16(ip + p) + 256; known = true; }
      else if (fcsId == 2) { fcs = ld32(ip + p); known = true; }
      else { fcs = ld64(ip + p); known = true; }
      if (single) window = fcs;
      if (dictID != 0 && dictID != ctxDictID) e = ZE_dictionary_wrong;             // :633 (ctxDictID = 0 without a dictionary, :2171)
      fi.fcs = fcs; fi.window = window;
      fi.flags = ((fhd >> 2) & 1 ? FI_CHECKSUM : 0) | (known ? FI_FCS_KNOWN : 0);
      fi.body_off = pos + fhs;
    }
  }
  if (e) { *result = zerr(e); fi.flags = FI_DONE; return false; }
  return true;
}

// =====================================================================================================
// Block header (GetcBlockSize :646-659 and the loop checks :2037-2042)
// =====================================================================================================
struct BlockHdr { u32 type, last, csize /* bytes of block content in src */, orig /* RLE length */; };
// rem = bytes left from the block header to the item's end.  Returns 0 or an error code.
ZB_HD u32 read_block_hdr(const u8* p, u32 rem, BlockHdr& b) {
  if (rem < 3) return ZE_srcSize_wrong;
  u32 h = ld24(p);
  b.last = h & 1; b.type = (h >> 1) & 3; b.orig = h >> 3;
  b.csize = b.type == 1 ? 1 : b.orig;
  if (b.type == 3) return ZE_corruption_detected;
  if (b.csize > rem - 3) return ZE_srcSize_wrong;
  return 0;
}

// =====================================================================================================
// Literals section header (DecodeLiteralsBlock :683-821, header part)
// =====================================================================================================
struct LitHdr {
  u32 type;       // 0 raw, 1 rle, 2 compressed, 3 repeat (treeless)
  u32 lhSize, litSize, litCSize;
  u32 single;     // single Huffman stream
  u32 consumed;   // bytes of the block taken by the literals section
};
// Returns 0 or an error code.  For type 3 the caller must additionally fail with dictionary_corrupted when no
// Huffman table is live; that check precedes the size checks in the reference (:696-699), so it is reported
// through *needs_table and must be resolved by the caller *before* looking at the returned code.
ZB_HD u32 read_lit_hdr(const u8* p, u32 srcSize, LitHdr& h, bool* needs_table) {
  *needs_table = false;
  if (srcSize < 3) return ZE_corruption_detected;                                  // :685
  h.type = p[0] & 3; u32 lhl = (p[0] >> 2) & 3; h.single = 0; h.litCSize = 0;
  if (h.type >= 2) {
    if (h.type == 3) *needs_table = true;
    if (srcSize < 5) return ZE_corruption_detected;                                // :699
    u32 lhc = ld32(p);
    if (lhl <= 1) { h.single = lhl == 0; h.lhSize = 3; h.litSize = (lhc >> 4) & 0x3FF; h.litCSize = (lhc >> 14) & 0x3FF; }
    else if (lhl == 2) { h.lhSize = 4; h.litSize = (lhc >> 4) & 0x3FFF; h.litCSize = lhc >> 18; }
    else { h.lhSize = 5; h.litSize = (lhc >> 4) & 0x3FFFF; h.litCSize = (lhc >> 22) + ((u32)p[4] << 10); }
    if (h.litSize > BLOCKSIZE_MAX) return ZE_corruption_detected;                  // :729
    if (h.litCSize + h.lhSize > srcSize) return ZE_corruption_detected;            // :730
    h.consumed = h.litCSize + h.lhSize;
    return 0;
  }
  if (lhl == 1) { h.lhSize = 2; h.litSize = ld16(p) >> 4; }
  else if (lhl == 3) { h.lhSize = 3; h.litSize = ld24(p) >> 4; }
  else { h.lhSize = 1; h.litSize = p[0] >> 3; }
  if (h.type == 0) {
    if (h.litSize + h.lhSize > srcSize) return ZE_corruption_detected;             // :774-776
    h.consumed = h.lhSize + h.litSize;
  } else {
    if (lhl == 3 && srcSize < 4) return ZE_corruption_detected;                    // :808
    if (h.litSize > BLOCKSIZE_MAX) return ZE_corruption_detected;                  // :811
    h.consumed = h.lhSize + 1;
  }
  return 0;
}

// =====================================================================================================
// Sequences section: count + mode byte (DecodeSeqHeaders :1110-1145)
// =====================================================================================================
// Returns 0 or error; *nbSeq, *modes (LL<<4|OF<<2|ML as 2-bit fields, 0 when nbSeq == 0), *hdr = bytes consumed
// up to and including the mode byte.
ZB_HD u32 read_seq_count(const u8* p, u32 srcSize, u32* nbSeq, u32* modes, u32* hdr) {
  if (srcSize < 1) return ZE_srcSize_wrong;
  u32 ip = 0, n = p[ip++];
  *modes = 0;
  if (n == 0) { *nbSeq = 0; *hdr = 1; return 0; }
  if (n > 0x7F) {
    if (n == 0xFF) { if (ip + 2 > srcSize) return ZE_srcSize_wrong; n = ld16(p + ip) + LONGNBSEQ; ip += 2; }
    else { if (ip >= srcSize) return ZE_srcSize_wrong; n = ((n - 0x80) << 8) + p[ip++]; }
  }
  *nbSeq = n;
  if (ip + 4 > srcSize) return ZE_srcSize_wrong;                                   // :1140
  u32 m = p[ip++];
  *modes = ((m >> 6) << 4) | (((m >> 4) & 3) << 2) | ((m >> 2) & 3);
  *hdr = ip;
  return 0;
}

// What k_parse learns from a frame's FIRST block for the kernels' per-class launches (p = the block header, rem = bytes
// left in the item).  *fewLiterals: compressed / treeless literals of at most 2 048 bytes (FI_SMALLHUF).  Returns the
// sequence-kernel class: 1 (FI_SEQ_A) when the block has at most aMax sequences, 2 (FI_SEQ_B) at most bMax, 0 = full-size
// tables (also when the block is raw / RLE or does not parse).  An encoder picks table logs of at most
// max(highbit(nbSeq - 1) - 2, highbit(largest code) + 2), i.e. <= 6 / 6 / 7 (LL / OF / ML) up to 512 sequences and <= 8 up
// to 2 048; a wrong guess is handed to the full-size kernel (SeqEmitter::defer).
ZB_HD u32 first_block_classes(const u8* p, u32 rem, u32 aMax, u32 bMax, bool* fewLiterals) {
  *fewLiterals = false;
  BlockHdr bh; LitHdr lh; bool needs;
  if (read_block_hdr(p, rem, bh) || bh.type != 2 || bh.csize >= BLOCKSIZE_MAX || read_lit_hdr(p + 3, bh.csize, lh, &needs)) return 0;
  *fewLiterals = lh.type >= 2 && lh.litSize <= 2048;
  u32 nbSeq, modes, hdr;
  if (read_seq_count(p + 3 + lh.consumed, bh.csize - lh.consumed, &nbSeq, &modes, &hdr)) return 0;
  return nbSeq <= aMax ? 1 : (nbSeq <= bMax ? 2 : 0);
}

// =====================================================================================================
// FSE normalized counts (ReadNCount, EntropyCommon.cs:79-188).  Index arithmetic in i32 relative to hb.
// =====================================================================================================
// NormT: anything indexable yielding s16& (plain pointer, or Strided<s16> for bank-interleaved shared memory)
template <class NormT>
ZB_HD u32 read_ncount(NormT norm, u32* maxSV, u32* tableLog, const u8* hb, u32 hbSize, u32* hdrBytes) {
  i32 ip = 0; const i32 iend = (i32)hbSize;
  if (hbSize < 4) return ZE_srcSize_wrong;
  u32 bitStream = ld32(hb);
  i32 nbBits = (i32)(bitStream & 0xF) + 5;
  if (nbBits > 15) return ZE_tableLog_tooLarge;
  bitStream >>= 4; i32 bitCount = 4;
  *tableLog = (u32)nbBits;
  i32 remaining = (1 << nbBits) + 1, threshold = 1 << nbBits;
  nbBits++;
  u32 charnum = 0; bool previous0 = false;
  while ((remaining > 1) & (charnum <= *maxSV)) {
    if (previous0) {
      u32 n0 = charnum;
      while ((bitStream & 0xFFFF) == 0xFFFF) {
        n0 += 24;
        if (ip < iend - 5) { ip += 2; bitStream = ld32(hb + ip) >> bitCount; }
        else { bitStream >>= 16; bitCount += 16; }
      }
      while ((bitStream & 3) == 3) { n0 += 3; bitStream >>= 2; bitCount += 2; }
      n0 += bitStream & 3; bitCount += 2;
      if (n0 > *maxSV) return ZE_maxSymbolValue_tooSmall;
      while (charnum < n0) norm[charnum++] = 0;
      if ((ip <= iend - 7) || (ip + (bitCount >> 3) <= iend - 4)) { ip += bitCount >> 3; bitCount &= 7; bitStream = ld32(hb + ip) >> bitCount; }
      else bitStream >>= 2;
    }
    {
      i32 max = (2 * threshold - 1) - remaining, count;
      if ((bitStream & (u32)(threshold - 1)) < (u32)max) { count = (i32)(bitStream & (u32)(threshold - 1)); bitCount += nbBits - 1; }
      else { count = (i32)(bitStream & (u32)(2 * threshold - 1)); if (count >= threshold) count -= max; bitCount += nbBits; }
      count--;
      remaining -= count < 0 ? -count : count;
      norm[charnum++] = (s16)count;
      previous0 = count == 0;
      while (remaining < threshold) { nbBits--; threshold >>= 1; }
      if ((ip <= iend - 7) || (ip + (bitCount >> 3) <= iend - 4)) { ip += bitCount >> 3; bitCount &= 7; }
      else { bitCount -= 8 * (iend - 4 - ip); ip = iend - 4; }
      bitStream = ld32(hb + ip) >> (bitCount & 31);
    }
  }
  if (remaining != 1) return ZE_corruption_detected;
  if (bitCount > 32) return ZE_corruption_detected;
  *maxSV = charnum - 1;
  ip += (bitCount + 7) >> 3;
  *hdrBytes = (u32)ip;
  return 0;
}

// =====================================================================================================
// Sequence-symbol decode tables (BuildFSETable :958-1034, rle :937-953, BuildSeqTable :1040-1079)
// =====================================================================================================
// Cell layout: one u16 per state (the reference's 8-byte SeqSymbol squeezed so that a frame's three tables take
// 2.5 KB of shared memory instead of 10):
//   bits 0..9   next-state base and state-bit count, jointly: ((base >> nb) << 1 | 1) << nb — base is always a
//               multiple of 1 << nb, so the lowest set bit marks nb and clearing it and halving gives base
//   bits 10..15 symbol (0..52); extra-bit count and base value come from the per-kind info tables below
ZB_HD u16 seq_cell(u32 nextState, u32 nbBits, u32 sym) { return (u16)(((((nextState >> nbBits) << 1) | 1) << nbBits) | (sym << 10)); }
ZB_HD u32 cell_nb(u32 low10) {
#if defined(__CUDA_ARCH__)
  return (u32)__ffs((int)low10) - 1;
#else
  return (u32)__builtin_ffs((int)low10) - 1;
#endif
}
ZB_HD u32 cell_base(u32 low10) { return (low10 & (low10 - 1)) >> 1; }
// The same decoding with a multiplication instead of a bit scan (the sequence loop's dependent chain): the low 10 bits
// are 2 * base + 2^nb, so the cell's lowest set bit is unit = 2^nb, and the high word of w * unit is the top nb bits of w.
// cell_next = the next state when w holds the state bits at its top.
ZB_HD u32 cell_unit(u32 cell) { return cell & (0u - cell); }
ZB_HD u32 cell_next(u32 cell, u32 unit, u32 w) {
  const u32 base = ((cell & 0x3FF) ^ unit) >> 1;
#if defined(__CUDA_ARCH__)
  u32 r; asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(unit), "r"(base)); return r;
#else
  return base + (u32)(((u64)w * unit) >> 32);
#endif
}

// base / extra-bit tables: ZStdInternal.cs:158-180, ZStdDecompress.cs:1081-1107
#if defined(__CUDACC__)
#define ZB_CONST_TABLE static __constant__
#else
#define ZB_CONST_TABLE static const
#endif
ZB_CONST_TABLE u8 kLLbits[36] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,1,1,1,1,2,2,3,3,4,6,7,8,9,10,11,12,13,14,15,16};
ZB_CONST_TABLE u8 kMLbits[53] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,
                                 1,1,1,1,2,2,3,3,4,4,5,7,8,9,10,11,12,13,14,15,16};
ZB_CONST_TABLE u32 kLLbase[36] = {0,1,2,3,4,5,6,7,8,9,10,11,12,13,14,15,16,18,20,22,24,28,32,40,48,64,0x80,0x100,0x200,0x400,0x800,0x1000,0x2000,0x4000,0x8000,0x10000};
ZB_CONST_TABLE u32 kMLbase[53] = {3,4,5,6,7,8,9,10,11,12,13,14,15,16,17,18,19,20,21,22,23,24,25,26,27,28,29,30,31,32,33,34,
                                  35,37,39,41,43,47,51,59,67,83,99,0x83,0x103,0x203,0x403,0x803,0x1003,0x2003,0x4003,0x8003,0x10003};
ZB_CONST_TABLE s16 kLLnorm[36] = {4,3,2,2,2,2,2,2,2,2,2,2,2,1,1,1,2,2,2,2,2,2,2,2,2,3,2,1,1,1,1,1,-1,-1,-1,-1};
ZB_CONST_TABLE s16 kMLnorm[53] = {1,4,3,2,2,2,2,2,2,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,
                                  1,1,1,1,1,1,1,1,1,1,1,1,1,1,-1,-1,-1,-1,-1,-1,-1};
ZB_CONST_TABLE s16 kOFnorm[29] = {1,1,1,1,1,1,2,2,2,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,-1,-1,-1,-1,-1};

ZB_HD u32 of_base(u32 code) { return code == 0 ? 0 : (code == 1 ? 1 : (1u << code) - 3); }   // :1088-1092

enum { KIND_LL = 0, KIND_OF = 1, KIND_ML = 2 };
ZB_HD u32 kind_nbadd(int kind, u32 sym) { return kind == KIND_LL ? kLLbits[sym] : (kind == KIND_ML ? kMLbits[sym] : sym); }

// per-symbol info word of the LL / ML kinds: base value | extra-bit count << 24
ZB_HD u32 ll_info(u32 sym) { return kLLbase[sym] | ((u32)kLLbits[sym] << 24); }
ZB_HD u32 ml_info(u32 sym) { return kMLbase[sym] | ((u32)kMLbits[sym] << 24); }

// Builds a decode table into cells[i*stride], i < (1<<tableLog).  `scratch` = 53 u16 of per-thread storage.
// The table must not be read through `cells` by anyone else meanwhile.
template <class NormT, class NextT>
ZB_HD void build_seq_table(u16* cells, u32 stride, NormT norm, u32 maxSV, u32 tableLog, NextT symbolNext) {
  u32 maxSV1 = maxSV + 1, tableSize = 1u << tableLog, high = tableSize - 1;
  for (u32 s = 0; s < maxSV1; s++) {
    if (norm[s] == -1) { cells[(high--) * stride] = (u16)s; symbolNext[s] = 1; }
    else symbolNext[s] = (u16)norm[s];
  }
  u32 mask = tableSize - 1, step = (tableSize >> 1) + (tableSize >> 3) + 3, pos = 0;   // Fse.cs:714-717
  for (u32 s = 0; s < maxSV1; s++)
    for (i32 i = 0; i < norm[s]; i++) {
      cells[pos * stride] = (u16)s;
      pos = (pos + step) & mask;
      while (pos > high) pos = (pos + step) & mask;
    }
  for (u32 u = 0; u < tableSize; u++) {
    u32 sym = cells[u * stride], next = symbolNext[sym]++;
    u32 nb = tableLog - highbit(next);
    cells[u * stride] = seq_cell(((next << nb) - tableSize) & 0x1FF, nb, sym);
  }
}

// One table descriptor of the sequences header.  mode: 0 predefined, 1 rle, 2 fse, 3 repeat.
// On success *log = table log now in force for this kind, *used = header bytes.  `cells/stride` is the
// lane-private table space; predefined tables live elsewhere (the caller switches pointers when *isDefault).
template <class NormT, class NextT>
// capLog: table log the space at `cells` can hold (the format's maximum unless a kernel instantiation keeps smaller tables):
// a larger, otherwise valid table is reported as ZB_TABLE_TOO_LARGE before anything is written.
ZB_HD u32 read_seq_table(u32 mode, int kind, const u8* p, u32 srcSize, u16* cells, u32 stride, u32* log, bool* isDefault,
                         bool haveRepeat, u32* used, NormT norm, NextT symbolNext, u32 capLog = 9) {
  const u32 maxSym = kind == KIND_LL ? MaxLL : (kind == KIND_ML ? MaxML : MaxOff);
  const u32 maxLog = kind == KIND_LL ? LLFSELog : (kind == KIND_ML ? MLFSELog : OffFSELog);
  *used = 0;
  switch (mode) {
    case 1: {
      if (srcSize == 0) return ZE_srcSize_wrong;
      u32 sym = p[0];
      if (sym > maxSym) return ZE_corruption_detected;
      cells[0] = seq_cell(0, 0, sym);
      *log = 0; *isDefault = false; *used = 1; return 0;
    }
    case 0: *isDefault = true; *log = kind == KIND_OF ? 5 : 6; return 0;
    case 3: return haveRepeat ? 0 : ZE_corruption_detected;
    default: {
      u32 max = maxSym, tl, h;
      u32 e = read_ncount(norm, &max, &tl, p, srcSize, &h);
      if (e) return ZE_corruption_detected;                                        // :1070
      if (tl > maxLog) return ZE_corruption_detected;                              // :1071
      if (tl > capLog) return ZB_TABLE_TOO_LARGE;
      build_seq_table(cells, stride, norm, max, tl, symbolNext);
      *log = tl; *isDefault = false; *used = h; return 0;
    }
  }
}

// =====================================================================================================
// Huffman weights and single-symbol table (ReadStats EntropyCommon.cs:198-269; FSE_decompress_wksp
// FseDecompress.cs:111-181,233-332; HUF_readDTableX2_wksp HufDecompress.cs:117-180)
// =====================================================================================================
// Workspace per Huffman table build.  weight/rank survive until the table has been filled; the FSE scratch is only
// live while compressed weights are decoded, so callers lend the (not yet filled) decode table for it.
struct HufBuildWk {
  u8 weight[256 + 4];
  u32 rank[16];
};
struct HufFseScratch {          // 1280 bytes
  s16 norm[256];
  u16 symbolNext[256];
  u32 fse[64];        // weight-FSE decode cells: newState | nbBits << 16 | symbol << 24
};

// FSE-compressed weights -> w[0..n).  Returns count, or 0xFFFFFFFF on error.  Mirrors the reference's
// two-state loop: symbols alternate between the states; once a read has crossed the stream start the other
// state's pending symbol is emitted and decoding stops (FseDecompress.cs:275-292).
// the same three arrays anywhere (the kernels lay them over memory that is idle while weights are read)
struct HufFseScratchRef { s16* norm; u16* symbolNext; u32* fse; };
template <class Scratch>
ZB_HD u32 fse_decode_weights(u8* w, u32 maxOut, const u8* src, u32 srcSize, Scratch& wk) {
  u32 maxSV = 255, tl, h;
  if (read_ncount(wk.norm, &maxSV, &tl, src, srcSize, &h)) return 0xFFFFFFFFu;
  if (tl > 6) return 0xFFFFFFFFu;                                                  // FseDecompress.cs:322 (maxLog 6)
  // BuildDTable, FseDecompress.cs:111-181
  u32 tableSize = 1u << tl, high = tableSize - 1;
  for (u32 s = 0; s <= maxSV; s++) {
    if (wk.norm[s] == -1) { wk.fse[high--] = s << 24; wk.symbolNext[s] = 1; }
    else wk.symbolNext[s] = (u16)wk.norm[s];
  }
  u32 mask = tableSize - 1, step = (tableSize >> 1) + (tableSize >> 3) + 3, pos = 0;
  for (u32 s = 0; s <= maxSV; s++)
    for (i32 i = 0; i < wk.norm[s]; i++) {
      wk.fse[pos] = s << 24;
      pos = (pos + step) & mask;
      while (pos > high) pos = (pos + step) & mask;
    }
  if (pos != 0) return 0xFFFFFFFFu;                                                // :165
  for (u32 u = 0; u < tableSize; u++) {
    u32 sym = wk.fse[u] >> 24, next = wk.symbolNext[sym]++;
    u32 nb = tl - highbit(next);
    wk.fse[u] = (((next << nb) - tableSize) & 0xFFFF) | (nb << 16) | (sym << 24);
  }
  // decode
  BitCursor c;
  if (!bc_init(c, src + h, srcSize - h)) return 0xFFFFFFFFu;
  i32 P = c.P;
  u32 s1, s2;
  { u64 win = bc_window64(c, P); s1 = tl ? (u32)(win >> (64 - tl)) : 0; P -= (i32)tl; }
  { u64 win = bc_window64(c, P); s2 = tl ? (u32)(win >> (64 - tl)) : 0; P -= (i32)tl; }
  // a negative P here is already "overflow"; the loop below then emits one symbol per state, as the reference does
  u32 n = 0;
  while (true) {
    if (n + 2 > maxOut) return 0xFFFFFFFFu;                                        // op > omax-2 -> dstSize_tooSmall
    { u32 cell = wk.fse[s1]; w[n++] = (u8)(cell >> 24); u32 nb = (cell >> 16) & 0xFF;
      u64 win = bc_window64(c, P); u32 low = nb ? (u32)(win >> (64 - nb)) : 0; P -= (i32)nb; s1 = (cell & 0xFFFF) + low; }
    if (P < 0) { w[n++] = (u8)(wk.fse[s2] >> 24); break; }
    if (n + 2 > maxOut) return 0xFFFFFFFFu;
    { u32 cell = wk.fse[s2]; w[n++] = (u8)(cell >> 24); u32 nb = (cell >> 16) & 0xFF;
      u64 win = bc_window64(c, P); u32 low = nb ? (u32)(win >> (64 - nb)) : 0; P -= (i32)nb; s2 = (cell & 0xFFFF) + low; }
    if (P < 0) { w[n++] = (u8)(wk.fse[s1] >> 24); break; }
  }
  return n;
}

// Parses the weight header at src and validates it.  On success returns 0 and sets *hdrBytes, *tableLog,
// *nbSym with wk.weight[0..nbSym), wk.rank[] = first cell index of each weight and slot[n] = how many earlier
// symbols share symbol n's weight — so that any lane can place any symbol's cells without a running count.
template <class Scratch>
ZB_HD u32 huf_read_weights(const u8* src, u32 srcSize, HufBuildWk& wk, Scratch& fs, u8* slot, u32* hdrBytes, u32* tableLog, u32* nbSym) {
  if (srcSize == 0) return ZE_srcSize_wrong;
  u32 iSize = src[0], oSize;
  if (iSize >= 128) {
    oSize = iSize - 127; iSize = (oSize + 1) / 2;
    if (iSize + 1 > srcSize) return ZE_srcSize_wrong;
    if (oSize >= 256) return ZE_corruption_detected;
    for (u32 n = 0; n < oSize; n += 2) { wk.weight[n] = src[1 + n / 2] >> 4; wk.weight[n + 1] = src[1 + n / 2] & 15; }
  } else {
    if (iSize + 1 > srcSize) return ZE_srcSize_wrong;
    oSize = fse_decode_weights(wk.weight, 255, src + 1, iSize, fs);
    if (oSize == 0xFFFFFFFFu) return ZE_corruption_detected;
  }
  for (u32 i = 0; i < 16; i++) wk.rank[i] = 0;
  u32 total = 0;
  for (u32 n = 0; n < oSize; n++) {
    u32 wv = wk.weight[n];
    if (wv >= HUF_LOG_MAX) return ZE_corruption_detected;
    slot[n] = (u8)wk.rank[wv];
    wk.rank[wv]++; total += (1u << wv) >> 1;
  }
  if (total == 0) return ZE_corruption_detected;
  u32 tl = highbit(total) + 1;
  if (tl > HUF_LOG_MAX) return ZE_corruption_detected;
  u32 rest = (1u << tl) - total, last = highbit(rest) + 1;
  if ((1u << highbit(rest)) != rest) return ZE_corruption_detected;
  wk.weight[oSize] = (u8)last; slot[oSize] = (u8)wk.rank[last]; wk.rank[last]++;
  if (wk.rank[1] < 2 || (wk.rank[1] & 1)) return ZE_corruption_detected;
  u32 next = 0;
  for (u32 n = 1; n < tl + 1; n++) { u32 cur = next; next += wk.rank[n] << (n - 1); wk.rank[n] = cur; }
  *hdrBytes = iSize + 1; *tableLog = tl; *nbSym = oSize + 1;
  return 0;
}

// Huffman decode cell: byte | nbBits << 8 (HufDecompress.cs:110-115)
// Fills table cells for symbols n = first, first+step, ... (so that several lanes can share the fill);
// rank starts must be advanced for *all* symbols in order, hence the full loop with a write predicate.
//
// The kernels keep 2^HUF_TABLE_LOG (11) cells per table — what every real encoder produces — so that more frames
// fit an SM's shared memory.  A log-12 table (legal for the reference, HufDecompress.cs:128) is folded: cell i stands
// for codes 2i and 2i+1.  Codes of 2..11 bits cover whole pairs (their first cell index is even because the weight-1
// symbols come first and their count is even, :389).  The 12-bit codes (weight 1) are the cells below count1/2:
// those get nbBits 12 and the two symbols of a pair go to side[2i], side[2i+1] (side: 256 bytes, only for log 12).
// dt must be 16-byte aligned: runs of 8 or more cells (power-of-two lengths at multiples of their length) are
// written as 16-byte vectors.
ZB_HD void huf_fill_cells(u16* dt, u32 start, u32 len, u16 cell) {
  if (len >= 8) {
    const u32 c2 = cell * 0x10001u;
    u32* p = (u32*)(dt + start);
    for (u32 u = 0; u < len / 2; u += 4) { p[u] = c2; p[u + 1] = c2; p[u + 2] = c2; p[u + 3] = c2; }
  } else for (u32 u = 0; u < len; u++) dt[start + u] = cell;
}
// longerThan: only the symbols whose code is longer than that many bits are entered (0 = all) — the kernels' full table
// in global memory only ever answers for codes the root table does not hold.
ZB_HD void huf_fill_table(u16* dt, u8* side, const HufBuildWk& wk, const u8* slot, u32 tableLog, u32 nbSym, u32 first, u32 step, u32 longerThan = 0) {
  const bool folded = tableLog > HUF_TABLE_LOG;
  for (u32 n = first; n < nbSym; n += step) {
    const u32 wv = wk.weight[n];
    if (!wv) continue;
    if (tableLog + 1 - wv <= longerThan) continue;
    const u32 len = 1u << (wv - 1), start = wk.rank[wv] + slot[n] * len;
    const u16 cell = (u16)(n | ((tableLog + 1 - wv) << 8));
    if (!folded) huf_fill_cells(dt, start, len, cell);
    else if (wv == 1) { side[start] = (u8)n; dt[start >> 1] = (u16)(12u << 8); }
    else huf_fill_cells(dt, start / 2, len / 2, cell);
  }
}

// Root table: 2^rootLog cells indexed by the next rootLog stream bits.  A code of at most that many bits owns whole
// root cells (its cell, as in the full table); the root cells under which only longer codes live hold HUF_LONG and the
// decoder looks those up in the full table (huf_fill_table with longerThan = rootLog).  The Huffman kernels live on how
// many frames an SM holds: rootLog 9 (1 KB per frame) for frames of few literals, whose table log is at most 9 with any
// known encoder; rootLog 11 otherwise (only the 12-bit codes of a log-12 table are then "long").
ZB_HD void huf_fill_root(u16* root, u32 rootLog, const HufBuildWk& wk, const u8* slot, u32 tableLog, u32 nbSym, u32 first, u32 step) {
  const u32 HUF_ROOT_LOG = rootLog;
  for (u32 n = first; n < nbSym; n += step) {
    const u32 wv = wk.weight[n];
    if (!wv) continue;
    const u32 cnt = 1u << (wv - 1), start = wk.rank[wv] + slot[n] * cnt, len = tableLog + 1 - wv;
    const u16 cell = (u16)(n | (len << 8));
    if (tableLog <= HUF_ROOT_LOG) huf_fill_cells(root, start << (HUF_ROOT_LOG - tableLog), cnt << (HUF_ROOT_LOG - tableLog), cell);
    else {
      const u32 sh = tableLog - HUF_ROOT_LOG;
      if (cnt >> sh) huf_fill_cells(root, start >> sh, cnt >> sh, cell);
      else root[start >> sh] = (u16)HUF_LONG;
    }
  }
}

// The root table of an existing full table (a dictionary's): cells first, first + step, ...
ZB_HD void huf_root_from_full(u16* root, u32 rootLog, const u16* full, u32 tableLog, u32 first, u32 step) {
  for (u32 i = first; i < (1u << rootLog); i += step) {
    if (tableLog <= rootLog) { root[i] = full[i >> (rootLog - tableLog)]; continue; }
    const u32 at = i << (tableLog - rootLog);                                      // first full-table index under this prefix
    const u32 c = full[tableLog > HUF_TABLE_LOG ? at >> 1 : at];                   // (a log-12 table is folded: cell j stands for 2j, 2j + 1)
    root[i] = (u16)((c >> 8) <= rootLog ? c : HUF_LONG);
  }
}

// =====================================================================================================
// Dictionary (ZSTD_decompress_insertDictionary :2449-2475, LoadEntropy :2375-2447, RefDictContent :2366-2373)
// =====================================================================================================
// Prepared once per context; every data frame then starts from it (ZSTD_decompressBegin_usingDict :2501-2507): the
// content is the window's prefix, and — for a dictionary with entropy tables — the Huffman table, the three sequence
// tables and the repeat offsets are what "repeat" / "treeless" modes of the first block refer to.
static const u32 MAGIC_DICT = 0xEC30A437u;
struct DictState {
  u32 present;            // 0: no dictionary
  u32 err;                // ZE_dictionary_corrupted when the entropy section is malformed: every data frame fails with it
  u32 dictID, hasEntropy;
  u32 rep[3];
  u32 hufLog;
  u32 log[3];             // KIND_LL, KIND_OF, KIND_ML
  u32 contentOff, contentSize;
  u32 pad;
  alignas(16) u16 cells[3][512];      // decode tables in the kernels' cell format (seq_cell), stride 1
  alignas(16) u16 huf[1u << HUF_TABLE_LOG];
  alignas(16) u8 hufSide[256];
};
// One thread.  norm / next: 53 entries each; slot: 256 bytes.
ZB_HD void dict_load(const u8* dict, u32 size, DictState& ds, HufBuildWk& wk, HufFseScratch& fs, u8* slot, s16* norm, u16* next) {
  ds.present = 1; ds.err = 0; ds.dictID = 0; ds.hasEntropy = 0; ds.rep[0] = 1; ds.rep[1] = 4; ds.rep[2] = 8; ds.hufLog = 0;
  ds.log[0] = ds.log[1] = ds.log[2] = 0; ds.contentOff = 0; ds.contentSize = size; ds.pad = 0;
  if (size < 8 || ld32(dict) != MAGIC_DICT) return;                                // pure content mode (:2451-2458)
  ds.dictID = ld32(dict + 4);
  ds.err = ZE_dictionary_corrupted;                                                // until the whole entropy section has been accepted
  if (size <= 8) return;
  u32 p = 8;
  {
    u32 hdr = 0, tl = 0, nbSym = 0;
    if (huf_read_weights(dict + p, size - p, wk, fs, slot, &hdr, &tl, &nbSym)) return;
    huf_fill_table(ds.huf, ds.hufSide, wk, slot, tl, nbSym, 0, 1);
    ds.hufLog = tl; p += hdr;
  }
  const int order[3] = {KIND_OF, KIND_ML, KIND_LL};
  for (int k = 0; k < 3; k++) {
    const int kind = order[k];
    const u32 maxSym = kind == KIND_LL ? MaxLL : (kind == KIND_ML ? MaxML : MaxOff);
    const u32 maxLog = kind == KIND_LL ? LLFSELog : (kind == KIND_ML ? MLFSELog : OffFSELog);
    u32 maxSV = maxSym, tl = 0, h = 0;
    if (read_ncount(norm, &maxSV, &tl, dict + p, size - p, &h)) return;
    if (maxSV > maxSym || tl > maxLog) return;
    build_seq_table(ds.cells[kind], 1, norm, maxSV, tl, next);
    ds.log[kind] = tl; p += h;
  }
  if (p + 12 > size) return;
  const u32 contentSize = size - (p + 12);
  for (int i = 0; i < 3; i++) { const u32 r = ld32(dict + p); p += 4; if (r == 0 || r >= contentSize) return; ds.rep[i] = r; }
  ds.contentOff = p; ds.contentSize = contentSize; ds.hasEntropy = 1; ds.err = 0;
}

}  // namespace zb
