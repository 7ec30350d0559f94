// zb_encode.cuh — per-thread body of the GPU zstd frame encoder (levels 1-3 and -7..-1).
//
// The reference repository ships no compressor (SURVEY.md §0 F1): what binds this code is the reference
// *decoder's* accept set — every structure written here is one that csharp/src/ZStdDecompress.cs,
// HufDecompress.cs, EntropyCommon.cs and FseDecompress.cs parse (citations at each writer) — plus the ratio
// band against libzstd at the same level.  The match finders follow the published zstd "fast" (levels 1-2) and
// "double-fast" (level 3) strategies: greedy parse over one (or a long+short pair of) position hash table(s),
// repeat-offset probing, step acceleration through incompressible runs.
//
// One GPU thread encodes one frame: frames are independent (the path shards by frame), a frame's blocks are
// sequentially dependent through the window, the repeat offsets and the hash tables.  Everything is
// __host__ __device__ so that tests/hostsim replays the same code on the CPU.
#pragma once
#include "zb_format.cuh"

namespace zb {



ZB_HD u64 rd64u(const u8* p) { return ld64(p); }
ZB_HD u32 rd32u(const u8* p) { return ld32(p); }

// position hash of the warp-parallel match finder (k_enc_match and its lock-step emulation in tests/hostsim) over the
// 8 bytes at a position: mls 8 hashes all of them, mls 5 / 6 the first 5 / 6
ZB_HD u32 hash64(u64 v, u32 hlog, u32 mls) {
  if (mls >= 8) return (u32)((v * 0xCF1BBCDCB7A56463ull) >> (64 - hlog));
  const u32 lo = (u32)v, hi = (u32)(v >> 32);                   // 5 / 6 bytes: two 32-bit multiplies do (ratio within 0.1 % of the 64-bit hash)
  return (lo * 2654435761u + (hi & (mls == 6 ? 0xFFFFu : 0xFFu)) * 2246822519u) >> (32 - hlog);
}

// Frame header of the encoder (mirrored by k_enc_entropy): single segment, Dictionary_ID field of 1 / 2 / 4 bytes when the
// id is not 0, content size of 1 / 2 / 4 bytes.  Returns its size; the caller has checked the room.
ZB_HD u32 enc_frame_header_size(u32 size, u32 dictID) {
  const u32 fcsCode = size < 256 ? 0 : (size < 65536 + 256 ? 1 : 2);
  const u32 didBytes = dictID == 0 ? 0 : (dictID < 256 ? 1 : (dictID < 65536 ? 2 : 4));
  return 4 + 1 + didBytes + (fcsCode == 0 ? 1 : (fcsCode == 1 ? 2 : 4));
}
ZB_HD u32 enc_frame_header(u8* dst, u32 size, int checksum, u32 dictID) {
  const u32 fcsCode = size < 256 ? 0 : (size < 65536 + 256 ? 1 : 2);
  const u32 didBytes = dictID == 0 ? 0 : (dictID < 256 ? 1 : (dictID < 65536 ? 2 : 4));
  dst[0] = 0x28; dst[1] = 0xB5; dst[2] = 0x2F; dst[3] = 0xFD;
  dst[4] = (u8)((fcsCode << 6) | (1u << 5) | (checksum ? 4 : 0) | (didBytes == 4 ? 3 : didBytes));
  u32 p = 5;
  for (u32 k = 0; k < didBytes; k++) dst[p++] = (u8)(dictID >> (8 * k));
  if (fcsCode == 0) dst[p++] = (u8)size;
  else if (fcsCode == 1) { const u32 v = size - 256; dst[p++] = (u8)v; dst[p++] = (u8)(v >> 8); }
  else { dst[p++] = (u8)size; dst[p++] = (u8)(size >> 8); dst[p++] = (u8)(size >> 16); dst[p++] = (u8)(size >> 24); }
  return p;
}



// ------------------------------------------------------------------------------------------------
// sequence store of one block
// ------------------------------------------------------------------------------------------------
struct SeqStore {
  u32* seqs; u32 n, cap;       // word0 = litLength, word1 = (matchLength - 3) | offCodeLow... see push
  u8* lits; u32 nlits;
};
ZB_HD void seq_get(const SeqStore& st, u32 i, u32& ll, u32& offBase, u32& mlm3) {
  u32 a = st.seqs[2 * i], b = st.seqs[2 * i + 1];
  ll = (a & 0xFFFF) | ((b >> 31) << 16);
  mlm3 = (a >> 16) | (((b >> 30) & 1) << 16);
  offBase = b & 0x3FFFFFFFu;
}



// ------------------------------------------------------------------------------------------------
// forward bit writer (the decoder reads it backwards: BitStream.cs:322-497).  Bits are appended LSB first.
// ------------------------------------------------------------------------------------------------
// Forward bit writer that stores whole aligned 32-bit words: p is 4-byte aligned, acc holds the nb pending bits
// (when the stream starts off alignment, the bytes already in memory before it ride along as the first pending
// bits and are stored back unchanged).  Contract: at most 32 bits are added between two bw_flush calls.
struct BitWriter { u8* p; u8* end; u64 acc; u32 nb; bool ovf; };
ZB_HD u32 bw_load32(const u8* p) { return (u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16) | ((u32)p[3] << 24); }
ZB_HD void bw_init(BitWriter& w, u8* p, u8* end) {
  const u32 a = (u32)((uintptr_t)p & 3);
  w.p = p - a; w.end = end; w.nb = 8 * a; w.ovf = false;
  w.acc = a ? (bw_load32(w.p) & ((1u << (8 * a)) - 1)) : 0;
}
ZB_HD void bw_add(BitWriter& w, u32 v, u32 n) { w.acc |= (u64)(v & ((n >= 32) ? 0xFFFFFFFFu : ((1u << n) - 1))) << w.nb; w.nb += n; }
ZB_HD void bw_flush(BitWriter& w) {   // keeps < 32 bits pending
  if (w.nb >= 32) {
    const u32 v = (u32)w.acc;
    if (w.p + 4 <= w.end) {
#if defined(__CUDA_ARCH__)
      *reinterpret_cast<u32*>(w.p) = v;
#else
      w.p[0] = (u8)v; w.p[1] = (u8)(v >> 8); w.p[2] = (u8)(v >> 16); w.p[3] = (u8)(v >> 24);
#endif
    } else { for (u32 k = 0; k < 4; k++) { if (w.p + k < w.end) w.p[k] = (u8)(v >> (8 * k)); else w.ovf = true; } }
    w.p += 4; w.acc >>= 32; w.nb -= 32;
  }
}
// end mark: a 1 bit, then zero padding (InitDStream locates it through the highest set bit of the last byte)
ZB_HD u8* bw_close(BitWriter& w) {
  bw_add(w, 1, 1); bw_flush(w);
  const u32 bytes = (w.nb + 7) >> 3;
  for (u32 k = 0; k < bytes; k++) { if (w.p + k < w.end) w.p[k] = (u8)(w.acc >> (8 * k)); else w.ovf = true; }
  w.p += bytes; w.nb = 0;
  return w.ovf ? nullptr : w.p;
}

// ------------------------------------------------------------------------------------------------
// FSE: normalisation, header, encoding table (accepted by ReadNCount EntropyCommon.cs:79-188 and
// BuildFSETable ZStdDecompress.cs:958-1034 / BuildDTable FseDecompress.cs:111-181)
// ------------------------------------------------------------------------------------------------
ZB_HD u32 fse_optimal_log(u32 maxLog, u32 total, u32 maxSym, u32 minus = 2) {
  u32 maxBitsSrc = highbit(total - 1) - minus;
  u32 minBitsSrc = highbit(total) + 1, minBitsSym = highbit(maxSym) + 2;
  u32 minBits = minBitsSrc < minBitsSym ? minBitsSrc : minBitsSym;
  u32 tl = maxLog;
  if (maxBitsSrc < tl) tl = maxBitsSrc;
  if (minBits > tl) tl = minBits;
  if (tl < 5) tl = 5;
  if (tl > 12) tl = 12;
  return tl;
}

// Normalised counts: integers n_s >= 1 for every present symbol with sum 1 << tableLog (what ReadNCount accepts:
// EntropyCommon.cs:79-188 only requires the counts to add up; the "-1 = less than one" form is never needed, a rare
// symbol simply gets one cell).
// Rounding rule: the cost of coding symbol s with n cells is count_s * log2(tableSize / n), so between floor(x) = n and
// n + 1 (x = the exact share) the better choice flips where x^2 = n (n + 1), the geometric mean — not at n + 1/2.  The
// rounded counts rarely add up exactly; the difference goes to / comes from the symbols with the most cells, where one
// cell more or less changes the code length least.  Returns false when one symbol holds every count (the caller
// writes an RLE table instead).
ZB_HD bool fse_normalize(s16* norm, u32 tableLog, const u32* count, u32 total, u32 maxSym) {
  const u32 tableSize = 1u << tableLog;
  const u64 step = ((u64)1 << 40) / total;               // total <= 2^17: count * step < 2^57
  const u32 shift = 40 - tableLog - 16;                  // share in Q16
  i32 sum = 0;
  for (u32 s = 0; s <= maxSym; s++) {
    if (count[s] == total) return false;
    if (count[s] == 0) { norm[s] = 0; continue; }
    const u64 x = (count[s] * step) >> shift;            // Q16, < 2^(tableLog + 16)
    u64 n = x >> 16;
    if (x * x > ((n * (n + 1)) << 32)) n++;
    if (n == 0) n = 1;
    norm[s] = (s16)n; sum += (i32)n;
  }
  i32 diff = (i32)tableSize - sum;                       // > 0: cells left over, < 0: too many handed out
  while (diff != 0) {
    u32 best = 0; s16 bestN = 0;
    for (u32 s = 0; s <= maxSym; s++) if (norm[s] > bestN) { bestN = norm[s]; best = s; }
    if (diff > 0) { norm[best] = (s16)(norm[best] + diff); diff = 0; }
    else {
      if (bestN <= 1) return false;                      // more present symbols than cells: cannot happen for tableLog >= log2(alphabet)
      const i32 take = -diff < bestN / 2 ? -diff : (bestN / 2 > 0 ? bestN / 2 : 1);   // at most half of a symbol's cells at a time
      norm[best] = (s16)(bestN - take); diff += take;
    }
  }
  return true;
}

// Header writer: the inverse of ReadNCount (EntropyCommon.cs:79-188), written against the reader.  The reader keeps
// `remaining` (cells not yet assigned, + 1) and `threshold` (the power of two above it): a count field stores n + 1 in
// nbBits - 1 bits when that value is below max = 2 * threshold - 1 - remaining, else in nbBits bits (values at or above
// threshold shifted up by max so that their low bits never look like a short field).  After a symbol with n = 0 the
// reader expects the length of the zero run that follows: 16 one-bits per 24 zeros, then the 2-bit value 3 per 3
// zeros, then the rest in 2 bits.  The table ends when every cell is assigned; the last byte is zero-padded.
// Returns bytes written or 0 when out of room.
ZB_HD u32 fse_write_ncount(u8* out, u32 cap, const s16* norm, u32 maxSym, u32 tableLog) {
  u64 acc = tableLog - 5; u32 nb = 4, op = 0;            // forward bit stream, least significant bit first
  i32 remaining = (1 << tableLog) + 1, threshold = 1 << tableLog, nbBits = (i32)tableLog + 1;
  u32 s = 0; bool afterZero = false;
  while (s <= maxSym && remaining > 1) {
    if (afterZero) {
      u32 run = 0;
      while (s + run <= maxSym && norm[s + run] == 0) run++;
      if (s + run > maxSym) return 0;                    // cells unassigned but no symbol left: not a valid distribution
      s += run;
      while (run >= 24) { acc |= (u64)0xFFFF << nb; nb += 16; run -= 24; while (nb >= 8) { if (op >= cap) return 0; out[op++] = (u8)acc; acc >>= 8; nb -= 8; } }
      while (run >= 3) { acc |= (u64)3 << nb; nb += 2; run -= 3; while (nb >= 8) { if (op >= cap) return 0; out[op++] = (u8)acc; acc >>= 8; nb -= 8; } }
      acc |= (u64)run << nb; nb += 2;
    }
    const i32 n = norm[s++];
    const i32 max = 2 * threshold - 1 - remaining;
    const i32 c = n + 1;                                 // stored value (n = -1 would store 0)
    if (c < max) { acc |= (u64)c << nb; nb += (u32)nbBits - 1; }
    else { acc |= (u64)(c < threshold ? c : c + max) << nb; nb += (u32)nbBits; }
    remaining -= n < 0 ? -n : n;
    if (remaining < 1) return 0;
    while (remaining < threshold) { nbBits--; threshold >>= 1; }
    afterZero = n == 0;
    while (nb >= 8) { if (op >= cap) return 0; out[op++] = (u8)acc; acc >>= 8; nb -= 8; }
  }
  if (remaining != 1) return 0;
  if (nb) { if (op >= cap) return 0; out[op++] = (u8)acc; }
  return op;
}

// encoding table: stateTable[tableSize] + per symbol (deltaNbBits, deltaFindState)
struct FseCTable { u16* stateTable; u32 tableLog; u32 deltaNbBits[64]; i32 deltaFindState[64]; };   // alphabets here have <= 53 symbols
ZB_HD void fse_build_ctable(FseCTable& ct, u16* stateTable, const s16* norm, u32 maxSym, u32 tableLog, u8* tableSymbol /* tableSize bytes */) {
  const u32 tableSize = 1u << tableLog, mask = tableSize - 1, step = (tableSize >> 1) + (tableSize >> 3) + 3;
  u32 cumul[258]; u32 high = tableSize - 1;
  ct.stateTable = stateTable; ct.tableLog = tableLog;
  cumul[0] = 0;
  for (u32 u = 1; u <= maxSym + 1; u++) {
    if (norm[u - 1] == -1) { cumul[u] = cumul[u - 1] + 1; tableSymbol[high--] = (u8)(u - 1); }
    else cumul[u] = cumul[u - 1] + (u32)norm[u - 1];
  }
  cumul[maxSym + 2] = tableSize + 1;
  { u32 pos = 0;
    for (u32 s = 0; s <= maxSym; s++)
      for (i32 i = 0; i < norm[s]; i++) { tableSymbol[pos] = (u8)s; pos = (pos + step) & mask; while (pos > high) pos = (pos + step) & mask; } }
  for (u32 u = 0; u < tableSize; u++) { u8 s = tableSymbol[u]; stateTable[cumul[s]++] = (u16)(tableSize + u); }
  { u32 total = 0;
    for (u32 s = 0; s <= maxSym; s++) {
      const i32 c = norm[s];
      if (c == 0) { ct.deltaNbBits[s] = ((tableLog + 1) << 16) - (1u << tableLog); ct.deltaFindState[s] = 0; }
      else if (c == -1 || c == 1) { ct.deltaNbBits[s] = (tableLog << 16) - (1u << tableLog); ct.deltaFindState[s] = (i32)total - 1; total++; }
      else {
        const u32 maxBitsOut = tableLog - highbit((u32)c - 1), minStatePlus = (u32)c << maxBitsOut;
        ct.deltaNbBits[s] = (maxBitsOut << 16) - minStatePlus; ct.deltaFindState[s] = (i32)total - c; total += (u32)c;
      }
    } }
}
ZB_HD void fse_build_ctable_rle(FseCTable& ct, u16* stateTable, u32 sym) {
  ct.stateTable = stateTable; ct.tableLog = 0; stateTable[0] = 0; stateTable[1] = 0;
  ct.deltaNbBits[sym] = 0; ct.deltaFindState[sym] = 0;
}
ZB_HD void fse_init_state(const FseCTable& ct, u32& state, u32 sym) {   // first symbol costs no bits
  const u32 nbBitsOut = (ct.deltaNbBits[sym] + (1u << 15)) >> 16;
  const u32 v = (nbBitsOut << 16) - ct.deltaNbBits[sym];
  state = ct.stateTable[(i32)(v >> nbBitsOut) + ct.deltaFindState[sym]];
}
ZB_HD void fse_encode(BitWriter& w, const FseCTable& ct, u32& state, u32 sym) {
  const u32 nbBitsOut = (state + ct.deltaNbBits[sym]) >> 16;
  bw_add(w, state, nbBitsOut);
  state = ct.stateTable[(i32)(state >> nbBitsOut) + ct.deltaFindState[sym]];
}
ZB_HD void fse_flush_state(BitWriter& w, const FseCTable& ct, u32 state) { bw_add(w, state, ct.tableLog); bw_flush(w); }

// ------------------------------------------------------------------------------------------------
// Huffman: length-limited code from a histogram, weight header, 1/4-stream encoding
// (accepted by ReadStats EntropyCommon.cs:198-269, HUF_readDTableX2 HufDecompress.cs:117-180,
//  4-stream layout HufDecompress.cs:266-307)
// ------------------------------------------------------------------------------------------------
struct HufCode { u16 val; u8 nbBits; };
struct HufEnc { HufCode code[256]; u8 weight[256]; u32 maxSym; u32 tableLog; };

// Builds code lengths <= maxBits for symbols with count > 0 (needs >= 2 distinct symbols).  Package-free
// heuristic: build an optimal tree with two queues over the sorted symbols, then repair over-long codes the
// way zstd's HUF_setMaxHeight does (pay back the Kraft debt on the longest cheap symbols).
// Working arrays of huf_build (4 KB): callers choose where they live (the GPU kernel lends shared memory).
// hash-table logs of the warp-parallel match finder (k_enc_match and its lock-step emulation in tests/hostsim)
// Table sizes of the match stage (log2 of u16 entries).  big: the launch holds chunks above one block (128 KiB): there a
// table of 2^12 entries forgets a position after ~4 KiB of input and the ratio falls out of the 3 % band against
// libzstd (tick records, level 1 at 256 KiB: -3.7 %, level 3 at 1 MiB: -4.1 %).  Level 1 then takes 2^13 entries (-2.0 %),
// level 3 a short table of 2^13 beside a long one of 2^12 (-0.7 % / -2.4 %; 24 KB, which still leaves 9 one-warp CTAs per
// SM: a GiB of 1 MiB chunks is 1 024 chunks and must not need a second wave).
// The negative (fast) levels take level 1's sizes: 2^12 entries as libzstd's hashLog 12 up to 128 KiB, 2^13 above.
ZB_HD u32 enc_hlog_long(int level, bool big) { return big ? (level >= 3 ? 12 : 13) : (level == 2 ? 13 : (level >= 3 ? 11 : 12)); }
ZB_HD u32 enc_hlog_short(int /*level*/, bool big) { return big ? 13 : 12; }
// Bytes the match stage's (short) hash covers: libzstd's minMatch, 6 at level 1, 5 at the negative levels (the ratio sweep
// of profiles/fast_levels_mls_sweep.jsonl) and at levels 2 and 3.
ZB_HD u32 enc_mls(int level) { return level == 1 ? 6 : 5; }
// Offset from the window start of the position lane l probes.  Levels 1-3: l * step.  Negative levels (accel): libzstd's fast
// loop, pairs of adjacent positions every `step` bytes, so lanes 2k and 2k + 1 probe k * step and k * step + 1; step starts at
// 1 + acceleration, which at acceleration 1 is every position.
ZB_HD u32 enc_probe_off(bool accel, u32 l, u32 step) { return accel ? (l >> 1) * step + (l & 1) : l * step; }

struct HufBuildScratch { u32 nodeCount[512]; u16 parent[512]; u16 order[256]; u8 depth[512]; };

// Stable sort of the used symbols by count ascending (ties: symbol ascending) -> order[0..n); returns n.
ZB_HD u32 huf_sort_symbols(u16* order, const u32* count, u32 maxSym) {
  u32 n = 0;
  for (u32 s = 0; s <= maxSym; s++) if (count[s]) order[n++] = (u16)s;
  for (u32 i = 1; i < n; i++) { u16 v = order[i]; u32 c = count[v]; u32 j = i; while (j > 0 && count[order[j - 1]] > c) { order[j] = order[j - 1]; j--; } order[j] = v; }
  return n;
}

// Code lengths and canonical values from he.weight[0..maxSym] (0 = unused) of a code of table log tl, matching the decoder's
// table fill: within a weight, symbols ascending; weights ascending start at rankStart (HufDecompress.cs:151-177):
// code value = cell index >> (tableLog - nbBits)
ZB_HD void huf_assign_codes(HufEnc& he, u32 maxSym, u32 tl) {
  he.tableLog = tl; he.maxSym = maxSym;
  u32 rankCount[16]; for (u32 i = 0; i < 16; i++) rankCount[i] = 0;
  for (u32 s = 0; s <= maxSym; s++) rankCount[he.weight[s]]++;
  u32 rankStart[16]; u32 nextStart = 0;
  for (u32 wv = 1; wv <= tl; wv++) { rankStart[wv] = nextStart; nextStart += rankCount[wv] << (wv - 1); }
  for (u32 s = 0; s <= maxSym; s++) {
    const u32 wv = he.weight[s];
    he.code[s].nbBits = wv ? (u8)(tl + 1 - wv) : 0;
    if (!wv) continue;
    he.code[s].val = (u16)(rankStart[wv] >> (wv - 1));
    rankStart[wv] += 1u << (wv - 1);
  }
}

// sc.order[0..n) holds the used symbols sorted as huf_sort_symbols does
ZB_HD bool huf_build_sorted(HufEnc& he, const u32* count, u32 n, u32 maxBits, HufBuildScratch& sc) {
  if (n < 2) return false;
  u16* const order = sc.order; u32* const nodeCount = sc.nodeCount; u16* const parent = sc.parent; u8* const depth = sc.depth;
  // two-queue Huffman: nodes 0..n-1 leaves (sorted), n..2n-2 internal
  for (u32 i = 0; i < n; i++) nodeCount[i] = count[order[i]];
  u32 leaf = 0, inner = n, next = n;
  while (next < 2 * n - 1) {
    u32 pick[2];
    for (int k = 0; k < 2; k++) {
      if (leaf < n && (inner >= next || nodeCount[leaf] <= nodeCount[inner])) pick[k] = leaf++; else pick[k] = inner++;
    }
    nodeCount[next] = nodeCount[pick[0]] + nodeCount[pick[1]];
    parent[pick[0]] = parent[pick[1]] = (u16)next; next++;
  }
  depth[2 * n - 2] = 0;
  for (i32 i = (i32)(2 * n - 3); i >= 0; i--) depth[i] = depth[parent[i]] + 1;
  // enforce the length limit: clamp, then repay the Kraft excess (in units of 2^-maxBits) by lengthening the
  // codes that are closest to the limit, and hand any overshoot back by shortening codes at the limit
  u32 largest = 0; for (u32 i = 0; i < n; i++) if (depth[i] > largest) largest = depth[i];
  if (largest > maxBits) {
    i64 debt = -((i64)1 << maxBits);
    for (u32 i = 0; i < n; i++) { if (depth[i] > maxBits) depth[i] = (u8)maxBits; debt += (i64)1 << (maxBits - depth[i]); }
    while (debt > 0) {
      i32 best = -1; i64 bestGain = 0;
      for (u32 i = 0; i < n; i++) {            // ascending count: the cheapest symbol of a depth comes first
        if (depth[i] >= maxBits) continue;
        const i64 gain = (i64)1 << (maxBits - depth[i] - 1);
        if (gain <= debt && gain > bestGain) { best = (i32)i; bestGain = gain; }
      }
      if (best < 0) {                          // every step overshoots: take the smallest one
        for (u32 i = 0; i < n; i++) if (depth[i] < maxBits) { const i64 gain = (i64)1 << (maxBits - depth[i] - 1); if (best < 0 || gain < bestGain) { best = (i32)i; bestGain = gain; } }
        if (best < 0) return false;
      }
      depth[best]++; debt -= bestGain;
    }
    while (debt < 0) {                         // refund one unit at a time: the most frequent code at the limit gets shorter
      i32 pick = -1;
      for (i32 i = (i32)n - 1; i >= 0; i--) if (depth[i] == maxBits) { pick = i; break; }
      if (pick < 0) return false;
      depth[pick]--; debt++;
    }
  }
  // the decoder derives the last weight, so the Kraft sum must be exactly 1 and tableLog = max depth
  u32 tl = 0; for (u32 i = 0; i < n; i++) if (depth[i] > tl) tl = depth[i];
  { u64 kraft = 0; for (u32 i = 0; i < n; i++) kraft += 1ull << (tl - depth[i]); if (kraft != (1ull << tl)) return false; }
  for (u32 s = 0; s < 256; s++) { he.code[s].nbBits = 0; he.code[s].val = 0; he.weight[s] = 0; }
  for (u32 i = 0; i < n; i++) he.weight[order[i]] = (u8)(tl + 1 - depth[i]);
  u32 maxSym = order[0];
  for (u32 i = 0; i < n; i++) if (order[i] > maxSym) maxSym = order[i];
  huf_assign_codes(he, maxSym, tl);
  return true;
}

// weight header: FSE-compressed weights when that is smaller, else 4-bit nibbles (needs maxSym <= 128 there)
ZB_HD u32 huf_write_header(u8* out, u32 cap, const HufEnc& he, u16* stateScratch, u8* symScratch) {
  const u32 nw = he.maxSym;   // weights of symbols 0..maxSym-1; the last one is implied
  if (nw == 0) return 0;
  // try FSE
  u32 fseSize = 0; alignas(4) u8 fseBuf[160];
  if (nw > 1) {
    u32 cnt[13]; for (u32 i = 0; i < 13; i++) cnt[i] = 0;
    u32 maxW = 0; for (u32 s = 0; s < nw; s++) { cnt[he.weight[s]]++; if (he.weight[s] > maxW) maxW = he.weight[s]; }
    bool single = false; for (u32 i = 0; i <= maxW; i++) if (cnt[i] == nw) single = true;
    if (!single && nw > 1) {
      u32 tl = fse_optimal_log(6, nw, maxW);
      if (tl > 6) tl = 6;
      s16 norm[13];
      if (fse_normalize(norm, tl, cnt, nw, maxW)) {
        u32 h = fse_write_ncount(fseBuf, 150, norm, maxW, tl);
        if (h) {
          FseCTable ct; fse_build_ctable(ct, stateScratch, norm, maxW, tl, symScratch);
          BitWriter w; bw_init(w, fseBuf + h, fseBuf + 150);
          // two interleaved states, last symbol first (decoder: FseDecompress.cs:233-295)
          i32 ip = (i32)nw; u32 s1, s2;
          if (nw & 1) { fse_init_state(ct, s1, he.weight[--ip]); fse_init_state(ct, s2, he.weight[--ip]); fse_encode(w, ct, s1, he.weight[--ip]); bw_flush(w); }
          else { fse_init_state(ct, s2, he.weight[--ip]); fse_init_state(ct, s1, he.weight[--ip]); }
          while (ip > 0) {
            fse_encode(w, ct, s2, he.weight[--ip]);
            if (ip > 0) fse_encode(w, ct, s1, he.weight[--ip]);
            bw_flush(w);
          }
          fse_flush_state(w, ct, s2); fse_flush_state(w, ct, s1);
          u8* e = bw_close(w);
          if (e) fseSize = (u32)(e - fseBuf);
        }
      }
    }
  }
  if (fseSize > 1 && fseSize < nw / 2 && fseSize < 128) {
    if (1 + fseSize > cap) return 0;
    out[0] = (u8)fseSize; for (u32 i = 0; i < fseSize; i++) out[1 + i] = fseBuf[i];
    return 1 + fseSize;
  }
  if (nw > 128) return 0;
  const u32 bytes = (nw + 1) / 2;
  if (1 + bytes > cap) return 0;
  out[0] = (u8)(128 + (nw - 1));
  for (u32 n = 0; n < nw; n += 2) out[1 + n / 2] = (u8)((he.weight[n] << 4) | (n + 1 < nw ? he.weight[n + 1] : 0));
  return 1 + bytes;
}

// one stream: symbols are written last-to-first so that the backward reader yields them in order
ZB_HD u32 huf_encode_stream(u8* out, u32 cap, const u8* src, u32 n, const HufEnc& he) {
  BitWriter w; bw_init(w, out, out + cap);
  for (i32 i = (i32)n - 1; i >= 0; i--) { const HufCode c = he.code[src[i]]; bw_add(w, c.val, c.nbBits); bw_flush(w); }
  u8* e = bw_close(w);
  return e ? (u32)(e - out) : 0;
}


// ------------------------------------------------------------------------------------------------
// sequences section (DecodeSeqHeaders :1110-1180, DecodeSequence :1473-1553)
// ------------------------------------------------------------------------------------------------
ZB_HD u32 ll_code(u32 ll) {
  if (ll < 16) return ll;
  if (ll < 64) { const u8 t[48] = {16,16,17,17,18,18,19,19,20,20,20,20,21,21,21,21,22,22,22,22,22,22,22,22,23,23,23,23,23,23,23,23,
                                   24,24,24,24,24,24,24,24,24,24,24,24,24,24,24,24}; return t[ll - 16]; }
  return highbit(ll) + 19;
}
ZB_HD u32 ml_code(u32 mlm3) {
  if (mlm3 < 32) return mlm3;
  if (mlm3 < 128) { const u8 t[96] = {32,32,33,33,34,34,35,35,36,36,36,36,37,37,37,37,38,38,38,38,38,38,38,38,39,39,39,39,39,39,39,39,40,40,40,40,40,40,40,40,40,40,40,40,40,40,40,40,41,41,41,41,41,41,41,41,41,41,41,41,41,41,41,41,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42,42};
                     return t[mlm3 - 32]; }
  return highbit(mlm3) + 36;
}

struct SeqKind { u32 maxSym, maxLog, defLog; const s16* defNorm; };

// chooses the table mode for one symbol kind and emits its description; returns the mode or 0xFF on failure
// count[] = histogram of the nbSeq codes of one kind (it is modified), lastCode = code of the last sequence
ZB_HD u32 enc_seq_table_counts(FseCTable& ct, u16* stateTable, u8* symScratch, u32* count, u32 lastCode, u32 nbSeq, const SeqKind& k, int level,
                               u8* out, u32 cap, u32* used) {
  u32 maxSym = k.maxSym; while (maxSym > 0 && !count[maxSym]) maxSym--;
  u32 most = 0; for (u32 s = 0; s <= maxSym; s++) if (count[s] > most) most = count[s];
  *used = 0;
  s16 norm[53];
  const bool defOk = maxSym <= (k.defLog == 5 ? 28u : k.maxSym);
  if (most == nbSeq) {
    if (defOk && nbSeq <= 2) { for (u32 s = 0; s <= k.maxSym; s++) norm[s] = s < (k.defLog == 5 ? 29u : k.maxSym + 1) ? k.defNorm[s] : 0;
      fse_build_ctable(ct, stateTable, norm, k.defLog == 5 ? 28 : k.maxSym, k.defLog, symScratch); return 0; }
    if (cap < 1) return 0xFF;
    out[0] = (u8)maxSym; *used = 1; fse_build_ctable_rle(ct, stateTable, maxSym); return 1;
  }
  if (defOk) {
    const u32 mult = 10 - (level <= 1 ? 1 : (level == 2 ? 1 : 2)), dynMin = ((1u << k.defLog) * mult) >> 3;
    if (nbSeq < dynMin || most < (nbSeq >> (k.defLog - 1))) {
      for (u32 s = 0; s <= k.maxSym; s++) norm[s] = s < (k.defLog == 5 ? 29u : k.maxSym + 1) ? k.defNorm[s] : 0;
      fse_build_ctable(ct, stateTable, norm, k.defLog == 5 ? 28 : k.maxSym, k.defLog, symScratch); return 0;
    }
  }
  u32 tl = fse_optimal_log(k.maxLog, nbSeq, maxSym);
  u32 total = nbSeq;
  if (count[lastCode] > 1) { count[lastCode]--; total--; }   // the last symbol costs no bits
  if (!fse_normalize(norm, tl, count, total, maxSym)) return 0xFF;
  u32 h = fse_write_ncount(out, cap, norm, maxSym, tl);
  if (!h) return 0xFF;
  *used = h;
  fse_build_ctable(ct, stateTable, norm, maxSym, tl, symScratch);
  return 2;
}

ZB_HD u32 enc_seq_count_header(u8* out, u32 nbSeq) {
  u32 op = 0;
  if (nbSeq < 128) out[op++] = (u8)nbSeq;
  else if (nbSeq < LONGNBSEQ) { out[op++] = (u8)((nbSeq >> 8) + 0x80); out[op++] = (u8)nbSeq; }
  else { out[op++] = 0xFF; out[op++] = (u8)(nbSeq - LONGNBSEQ); out[op++] = (u8)((nbSeq - LONGNBSEQ) >> 8); }
  return op;
}


ZB_HD SeqKind seq_kind(int kind) {
  if (kind == KIND_LL) return SeqKind{MaxLL, LLFSELog, 6, kLLnorm};
  if (kind == KIND_OF) return SeqKind{MaxOff, OffFSELog, 5, kOFnorm};
  return SeqKind{MaxML, MLFSELog, 6, kMLnorm};
}





// ------------------------------------------------------------------------------------------------
// encoder-side dictionary (zstdb200_compress*_using_dict): prepared once per zstdb200_load_dictionary on the host,
// copied to every device as one block  [EncDict][three match tables][content + 64 bytes of read slack]
// ------------------------------------------------------------------------------------------------
// Match tables of the dictionary content: 2^ENC_DICT_HLOG u32 content positions each, ENC_DICT_EMPTY where no position
// hashes.  One table per hash the match stage uses: mls 6 (level 1), mls 5 (level 2, and level 3's short table), the
// 8-byte long hash (level 3).  They are read-only and shared by every warp, so they can be larger than the per-warp
// chunk tables, but larger is not better: in a ratio sweep of the lock-step emulation (256 x 4 KiB log messages, 32 KiB
// trained dictionary, profiles/dict_match_table_sweep.jsonl) 2^12 .. 2^16 entries give 4.715 / 4.695 / 4.685 / 4.678 / 4.675
// at level 1 and 4.523 .. 4.463 at level 2 (a greedy parse takes the first hit: fewer, more recent dictionary positions
// leave more to the cheaper in-chunk matches); level 3 is flat (4.686 .. 4.679).  2^12 is also the smallest (48 KB).
#define ENC_DICT_HLOG 12
static constexpr u32 ENC_DICT_EMPTY = 0xFFFFFFFFu;
enum { EDT_MLS6 = 0, EDT_MLS5 = 1, EDT_LONG = 2 };
struct alignas(16) EncDict {
  u32 err;               // ZE_dictionary_corrupted when the entropy section is malformed: every item fails with it
  u32 dictID;            // written into the frame header when not 0 (a raw-content dictionary has id 0)
  u32 contentSize;       // bytes of content the match tables index (0 when err)
  u32 rep[3];            // the repeat offsets a frame starts from (1, 4, 8 for a raw-content dictionary)
  u32 hasEntropy;        // the tables below are the dictionary's (magic 0xEC30A437): what a frame's first block may reuse
  u32 pad;
  // Huffman encoding table from the dictionary's weights (the canonical codes huf_fill_table decodes), and the three FSE
  // compression tables from its normalized counts (KIND_LL, KIND_OF, KIND_ML; seqCt[k].stateTable is set where it is used:
  // seqState[k] at the address the reader sees)
  HufEnc huf;
  FseCTable seqCt[3];
  s16 seqNorm[3][64];
  u32 seqMaxSV[3], pad2;
  u16 seqState[3][512];
};
ZB_HD size_t enc_dict_bytes(u32 contentSize) { return sizeof(EncDict) + 3 * ((size_t)4 << ENC_DICT_HLOG) + contentSize + 64; }
ZB_HD const u32* enc_dict_table(const EncDict* d, int which) { return reinterpret_cast<const u32*>(d + 1) + ((size_t)which << ENC_DICT_HLOG); }
ZB_HD const u8* enc_dict_content(const EncDict* d) { return reinterpret_cast<const u8*>(d + 1) + 3 * ((size_t)4 << ENC_DICT_HLOG); }

// Fills the block at `out` (enc_dict_bytes(ds.err ? 0 : ds.contentSize) bytes) from the dictionary bytes (size of them, readable
// 64 bytes further) and what dict_load parsed of them (the decoder's preparation: id, content range, repeat offsets, validity of
// the entropy section).  An entropy dictionary's Huffman weights and normalized counts are read again (huf_read_weights,
// read_ncount: dict_load keeps only the decode tables) and turned into encoding tables.  Every content position whose 8 bytes
// lie inside the content is entered into the match tables in ascending order: the last one of a hash wins.
// Scratch: tableSymbol 512 bytes, slot 256 bytes.
ZB_HD void enc_dict_prepare(const u8* dict, u32 size, const DictState& ds, EncDict* out, HufBuildWk& wk, HufFseScratch& fs, u8* slot, u8* tableSymbol) {
  out->err = ds.err; out->dictID = ds.dictID; out->contentSize = ds.err ? 0 : ds.contentSize;
  for (int i = 0; i < 3; i++) out->rep[i] = ds.rep[i];
  out->hasEntropy = !ds.err && ds.hasEntropy; out->pad = 0; out->pad2 = 0;
  for (u32 s = 0; s < 256; s++) { out->huf.code[s].val = 0; out->huf.code[s].nbBits = 0; out->huf.weight[s] = 0; }
  out->huf.maxSym = 0; out->huf.tableLog = 0;
  for (int k = 0; k < 3; k++) {
    out->seqCt[k] = FseCTable(); out->seqMaxSV[k] = 0;
    for (u32 s = 0; s < 64; s++) out->seqNorm[k][s] = 0;
    for (u32 i = 0; i < 512; i++) out->seqState[k][i] = 0;
  }
  if (out->hasEntropy) {
    u32 p = 8, hdr = 0, tl = 0, nbSym = 0;
    huf_read_weights(dict + p, size - p, wk, fs, slot, &hdr, &tl, &nbSym);      // accepted by dict_load: cannot fail here
    for (u32 s = 0; s < nbSym; s++) out->huf.weight[s] = wk.weight[s];
    huf_assign_codes(out->huf, nbSym - 1, tl);
    p += hdr;
    const int order[3] = {KIND_OF, KIND_ML, KIND_LL};
    for (int o = 0; o < 3; o++) {
      const int kind = order[o];
      u32 maxSV = kind == KIND_LL ? MaxLL : (kind == KIND_ML ? MaxML : MaxOff), stl = 0, h = 0;
      read_ncount(out->seqNorm[kind], &maxSV, &stl, dict + p, size - p, &h);
      fse_build_ctable(out->seqCt[kind], out->seqState[kind], out->seqNorm[kind], maxSV, stl, tableSymbol);
      out->seqCt[kind].stateTable = nullptr;
      out->seqMaxSV[kind] = maxSV; p += h;
    }
  }
  u32* const t = const_cast<u32*>(enc_dict_table(out, 0));
  for (u32 i = 0; i < 3u << ENC_DICT_HLOG; i++) t[i] = ENC_DICT_EMPTY;
  u8* const content = const_cast<u8*>(enc_dict_content(out));
  const u32 n = out->contentSize;
  for (u32 i = 0; i < n; i++) content[i] = dict[ds.contentOff + i];
  for (u32 i = 0; i < 64; i++) content[n + i] = 0;
  u32* const t6 = t + ((u32)EDT_MLS6 << ENC_DICT_HLOG); u32* const t5 = t + ((u32)EDT_MLS5 << ENC_DICT_HLOG); u32* const tl = t + ((u32)EDT_LONG << ENC_DICT_HLOG);
  for (u32 q = 0; q + 8 <= n; q++) {
    const u64 v = ld64(content + q);
    t6[hash64(v, ENC_DICT_HLOG, 6)] = q; t5[hash64(v, ENC_DICT_HLOG, 5)] = q; tl[hash64(v, ENC_DICT_HLOG, 8)] = q;
  }
}

// Estimated cost in 1/256 bits of coding count[s] symbols s <= maxSym with the FSE table ct (libzstd's ZSTD_fseBitCost per
// symbol, from the table's deltaNbBits; an RLE table costs nothing).
ZB_HD u64 fse_cost256(const FseCTable& ct, const u32* count, u32 maxSym) {
  if (ct.tableLog == 0) return 0;
  const u32 tableSize = 1u << ct.tableLog;
  u64 bits = 0;
  for (u32 s = 0; s <= maxSym; s++) {
    if (!count[s]) continue;
    const u32 d = ct.deltaNbBits[s], minNb = d >> 16, threshold = (minNb + 1) << 16;
    bits += (u64)count[s] * (((minNb + 1) << 8) - (((threshold - (d + tableSize)) << 8) >> ct.tableLog));
  }
  return bits;
}

// enc_seq_table_counts, and for the first block of a frame with an entropy dictionary (ed != null) repeat mode (3) with the
// dictionary's table when every code present has a non-zero probability there (and is at most its maxSV) and its estimated
// bits are fewer than those of the mode chosen without it (its table description included).  count[] as for
// enc_seq_table_counts.
ZB_HD u32 enc_seq_table_counts_dict(FseCTable& ct, u16* stateTable, u8* symScratch, u32* count, u32 lastCode, u32 nbSeq, const SeqKind& k,
                                    int level, u8* out, u32 cap, u32* used, const EncDict* ed, int kind) {
  const u32 cLast = count[lastCode];
  const u32 m = enc_seq_table_counts(ct, stateTable, symScratch, count, lastCode, nbSeq, k, level, out, cap, used);
  if (!ed || m == 0xFF) return m;
  count[lastCode] = cLast;
  u32 maxSym = k.maxSym; while (maxSym > 0 && !count[maxSym]) maxSym--;
  if (maxSym > ed->seqMaxSV[kind]) return m;
  for (u32 s = 0; s <= maxSym; s++) if (count[s] && ed->seqNorm[kind][s] == 0) return m;
  if (fse_cost256(ed->seqCt[kind], count, maxSym) >= fse_cost256(ct, count, maxSym) + ((u64)*used << 11)) return m;
  ct = ed->seqCt[kind]; ct.stateTable = const_cast<u16*>(ed->seqState[kind]); *used = 0;
  return 3;
}

// Treeless literals (type 3) with the dictionary's Huffman code for the first block of a frame: when every literal present has
// a code there and the estimated stream bits are fewer than those of the fresh code `he` plus its header of hdrBytes.
ZB_HD bool huf_dict_better(const HufEnc& dictHuf, const HufEnc& he, u32 hdrBytes, const u32* count) {
  u64 dictBits = 0, freshBits = (u64)hdrBytes * 8;
  for (u32 s = 0; s < 256; s++) {
    if (!count[s]) continue;
    if (!dictHuf.code[s].nbBits) return false;
    dictBits += (u64)count[s] * dictHuf.code[s].nbBits; freshBits += (u64)count[s] * he.code[s].nbBits;
  }
  return dictBits < freshBits;
}

}  // namespace zb
