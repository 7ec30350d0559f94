// zb_dict_train.cuh — dictionary training (zstdb200_train_dictionary): the parts shared by the kernels, the host and the
// CPU emulation in tests/hostsim/dict_train.cpp.
//
// Content selection reproduces libzstd 1.5.5's fastCover trainer (ZDICT_trainFromBuffer_fastCover and the k search of
// ZDICT_optimizeTrainFromBuffer_fastCover): the d-mer hash, the sampling of the frequency pass, the epoch rule and the segment
// score.  The entropy section is built from this library's own match stage (k_enc_match over the first block of each
// finalize sample) with ZDICT_analyzeEntropy's rules: every symbol counted once more, Huffman at most 11 bits, FSE logs
// OF 8 / ML 9 / LL 9, repeat offsets 1, 4, 8.
#pragma once
#include "zb_encode.cuh"

namespace zb {

#define DT_DICT_MIN 256u              // ZDICT_DICTSIZE_MIN
#define DT_MAX_F 24u
#define DT_ZERO_SCORE_RUN 10u         // selection stops after this many consecutive epochs without a scoring segment
#define DT_SEARCH_KS 5u
#define DT_LOOKBACK 2048u             // the k_dt_prev window: > L - 1 for every k of the search grid and every fixed k <= DT_MAX_K
#define DT_MAX_K 2048u

// ZDICT_trainFromBuffer's k grid: kMinK 50 .. kMaxK 2000 in 4 steps of (2000 - 50) / 4
ZB_HD u32 dt_search_k(u32 i) { return 50u + 487u * i; }

// fastCover acceleration: share of the training samples whose first block feeds the entropy statistics (percent), and the
// positions the frequency pass skips between two counted ones (FASTCOVER_defaultAccelParameters)
ZB_HD u32 dt_accel_finalize(u32 accel) {
  switch (accel) { case 2: return 50; case 3: return 34; case 4: return 25; case 5: return 20; case 6: return 17;
                   case 7: return 14; case 8: return 13; case 9: return 11; case 10: return 10; default: return 100; }
}
ZB_HD u32 dt_accel_skip(u32 accel) { return accel >= 1 ? accel - 1 : 0; }

// FASTCOVER_hashPtrToIndex: zstd's ZSTD_hash6Ptr (d = 6) or ZSTD_hash8Ptr over the little-endian 8 bytes at p, f bits
ZB_HD u32 dt_hash(const u8* p, u32 f, u32 d) {
  const u64 v = ld64(p);
  if (d == 6) return (u32)(((v << 16) * 227718039650203ull) >> (64 - f));
  return (u32)((v * 0xCF1BBCDCB7A56463ull) >> (64 - f));
}

// COVER_computeEpochs with passes = 1
struct DtEpochs { u32 num, size; };
ZB_HD DtEpochs dt_epochs(u32 capacity, u32 nbDmers, u32 k) {
  DtEpochs e;
  e.num = capacity / k > 1 ? capacity / k : 1;
  e.size = nbDmers / e.num;
  if (e.size >= 10 * k) return e;
  e.size = 10 * k < nbDmers ? 10 * k : nbDmers;
  e.num = e.size ? nbDmers / e.size : 0;
  return e;
}

// XXH64 with seed 0, one thread (ZDICT's dictionary id is taken from it)
ZB_HD u64 dt_rotl(u64 x, u32 r) { return (x << r) | (x >> (64 - r)); }
ZB_HD u64 dt_xxh64(const u8* p, u64 len) {
  const u64 P1 = 0x9E3779B185EBCA87ull, P2 = 0xC2B2AE3D27D4EB4Full, P3 = 0x165667B19E3779F9ull, P4 = 0x85EBCA77C2B2AE63ull,
            P5 = 0x27D4EB2F165667C5ull;
  auto round = [&](u64 acc, u64 in) { acc += in * P2; acc = dt_rotl(acc, 31); return acc * P1; };
  u64 h; u64 i = 0;
  if (len >= 32) {
    u64 v1 = P1 + P2, v2 = P2, v3 = 0, v4 = 0 - P1;
    for (; i + 32 <= len; i += 32) { v1 = round(v1, ld64(p + i)); v2 = round(v2, ld64(p + i + 8)); v3 = round(v3, ld64(p + i + 16)); v4 = round(v4, ld64(p + i + 24)); }
    h = dt_rotl(v1, 1) + dt_rotl(v2, 7) + dt_rotl(v3, 12) + dt_rotl(v4, 18);
    const u64 vs[4] = {v1, v2, v3, v4};
    for (int k = 0; k < 4; k++) { h ^= round(0, vs[k]); h = h * P1 + P4; }
  } else h = P5;
  h += len;
  for (; i + 8 <= len; i += 8) { h ^= round(0, ld64(p + i)); h = dt_rotl(h, 27) * P1 + P4; }
  if (i + 4 <= len) { h ^= (u64)ld32(p + i) * P1; h = dt_rotl(h, 23) * P2 + P3; i += 4; }
  for (; i < len; i++) { h ^= (u64)p[i] * P5; h = dt_rotl(h, 11) * P1; }
  h ^= h >> 33; h *= P2; h ^= h >> 29; h *= P3; h ^= h >> 32;
  return h;
}

// Symbol statistics of the match stage over the finalize samples: literal bytes and the LL / ML / OF codes of every sequence
struct DtStats { u32 lit[256], ll[MaxLL + 1], ml[MaxML + 1], of[32]; };

ZB_HD void dt_flat_lit(u32* lit) {   // ZDICT_flatLit
  for (u32 s = 1; s < 256; s++) lit[s] = 2;
  lit[0] = 4; lit[253] = 1; lit[254] = 1;
}

// Work areas of dt_write_header (about 9 KB): callers choose where they live
struct DtHeaderScratch { HufEnc he; HufBuildScratch hb; u16 state[514 + 2]; u8 sym[512 + 16]; s16 norm[64]; };

// The dictionary header and entropy section: magic 0xEC30A437, dictID, Huffman weights, OF / ML / LL normalized counts and the
// repeat offsets 1, 4, 8.  st is modified (every symbol counted once more, as ZDICT_analyzeEntropy starts its counts at 1).
// selSize: bytes of selected content (it sets the largest offset code a dictionary of it can need).  out needs DT_DICT_MIN
// bytes.  Returns the header size, 0 when a table cannot be written (cannot happen for counts that every symbol has).
ZB_HD u32 dt_write_header(u8* out, u32 dictID, DtStats& st, u32 selSize, DtHeaderScratch& w) {
  const u32 cap = DT_DICT_MIN;
  out[0] = 0x37; out[1] = 0xA4; out[2] = 0x30; out[3] = 0xEC;
  out[4] = (u8)dictID; out[5] = (u8)(dictID >> 8); out[6] = (u8)(dictID >> 16); out[7] = (u8)(dictID >> 24);
  u32 op = 8;
  u32 ofMax = highbit(selSize + (128u << 10));
  for (u32 s = ofMax + 1; s < 32; s++) if (st.of[s]) ofMax = s;
  for (u32 s = 0; s < 256; s++) st.lit[s]++;
  for (u32 s = 0; s <= MaxLL; s++) st.ll[s]++;
  for (u32 s = 0; s <= MaxML; s++) st.ml[s]++;
  for (u32 s = 0; s <= ofMax; s++) st.of[s]++;
  // Huffman: weights of all 256 symbols; a distribution whose header cannot be written is flattened as ZDICT does
  u32 h = 0;
  for (int attempt = 0; attempt < 2 && !h; attempt++) {
    if (attempt) dt_flat_lit(st.lit);
    const u32 n = huf_sort_symbols(w.hb.order, st.lit, 255);
    if (huf_build_sorted(w.he, st.lit, n, 11, w.hb)) h = huf_write_header(out + op, cap - op, w.he, w.state, w.sym);
  }
  if (!h) return 0;
  op += h;
  const u32* counts[3] = {st.of, st.ml, st.ll};
  const u32 maxSym[3] = {ofMax, MaxML, MaxLL}, logs[3] = {OffFSELog, MLFSELog, LLFSELog};
  for (int k = 0; k < 3; k++) {
    u32 total = 0;
    for (u32 s = 0; s <= maxSym[k]; s++) total += counts[k][s];
    if (!fse_normalize(w.norm, logs[k], counts[k], total, maxSym[k])) return 0;
    const u32 c = fse_write_ncount(out + op, cap - op, w.norm, maxSym[k], logs[k]);
    if (!c) return 0;
    op += c;
  }
  if (op + 12 > cap) return 0;
  const u32 rep[3] = {1, 4, 8};
  for (int k = 0; k < 3; k++) for (int b = 0; b < 4; b++) out[op++] = (u8)(rep[k] >> (8 * b));
  return op;
}

// ZDICT's dictionary id rule: XXH64 of the whole selection, mod 2^31 - 32768, + 32768
ZB_HD u32 dt_dict_id(const u8* sel, u32 selSize) { return (u32)(dt_xxh64(sel, selSize) % ((1ull << 31) - 32768)) + 32768u; }

// ZDICT_finalizeDictionary's layout: header, zero padding up to the largest repeat offset (8), content.  Content that does not
// fit beside the header loses its end, as in libzstd 1.5.5 (there the segments selected first sit).  Returns the dictionary size.
ZB_HD u32 dt_assemble(u8* out, u32 capacity, const u8* hdr, u32 hSize, const u8* sel, u32 selSize) {
  u32 keep = selSize;
  if (hSize + keep > capacity) keep = capacity - hSize;
  const u32 pad = keep < 8 ? 8 - keep : 0;
  for (u32 i = 0; i < hSize; i++) out[i] = hdr[i];
  for (u32 i = 0; i < pad; i++) out[hSize + i] = 0;
  for (u32 i = 0; i < keep; i++) out[hSize + pad + i] = sel[i];
  return hSize + pad + keep;
}

// The raw-content dictionary the match stage gathers statistics with: the selection itself, id 0, repeat offsets 1, 4, 8
ZB_HD void dt_raw_dict_state(DictState& ds, u32 size) {
  ds.present = 1; ds.err = 0; ds.dictID = 0; ds.hasEntropy = 0; ds.rep[0] = 1; ds.rep[1] = 4; ds.rep[2] = 8; ds.hufLog = 0;
  ds.log[0] = ds.log[1] = ds.log[2] = 0; ds.contentOff = 0; ds.contentSize = size; ds.pad = 0;
}

}  // namespace zb
