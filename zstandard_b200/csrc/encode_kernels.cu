// encode_kernels.cu — sm_100a kernels of the batched zstd frame encoder.
//
//   k_enc_match<DFAST, DICT, ACCEL>      (DICT: also against the context's dictionary; ACCEL: the negative levels; see the kernel)
//                      : warp / block    match finder: 32 consecutive (or strided) positions per step, one per lane;
//                                        position hash table(s) of u16 entries in per-warp global scratch (L1 / L2
//                                        resident; 32 one-warp CTAs per SM) or, for the concurrent slices of a host
//                                        batch, in shared memory; in-window duplicate
//                                        hashes resolved with __match_any_sync, candidates verified in parallel, the
//                                        first hit wins (greedy parse), match length by warp ballot; sequence store
//                                        and literals go to HBM scratch
//   k_enc_entropy      : warp / frame    literals: histogram, Huffman code (symbols sorted across the warp), 4 streams on
//                                        4 lanes; sequences: codes + histograms in parallel, FSE tables (lane 0), the
//                                        three FSE state chains on three lanes and the bitstream packed by all lanes
//                                        through a warp prefix sum of field widths; block + frame assembly
//   k_enc_xxh          : 4 lanes / frame XXH64 content checksum appended to the frame (xxh_device.cuh)
//
// Frames are independent, so there is no inter-warp communication.  HBM scratch of the match stage is addressed
// from src_off (no scan): literals of item f at lit + src_off[f] + 64 f, sequences (8-byte entries) at
// seq + src_off[f]/4 + 64 (src_off[f] >> 17) + 128 f, block metadata at meta + (src_off[f] >> 17) + f.
#include "encode_kernels.cuh"
#include "zb_encode.cuh"
#include "zb_encode_warp.cuh"
#include "xxh_device.cuh"
#include <stdio.h>

namespace zb {

#define ENC_PRIME 16384u   // bytes before a block that prime its match tables (multiple of 32, <= BLOCKSIZE_MAX)

struct BlockMeta { u32 nseq, nlits; };
static constexpr u32 kGtabStride = 24 * 1024;   // bytes of global table space per match-stage warp: the largest tables of enc_hlog_*
static constexpr u32 kGtabWarpsPerSm = 32;      // one-warp CTAs resident per SM (the hardware's CTA limit)

__device__ __forceinline__ u8* lit_base(const EncodeArgs& a, const EncodeScratch& s, u32 f) { return s.lit + a.src_off[f] + 64ull * (a.item_base + f); }
__device__ __forceinline__ u32* seq_base(const EncodeArgs& a, const EncodeScratch& s, u32 f) {
  const u64 o = a.src_off[f];
  return s.seq + 2 * (o / 4 + 64 * (o >> 17) + 128ull * (a.item_base + f));
}
__device__ __forceinline__ BlockMeta* meta_base(const EncodeArgs& a, const EncodeScratch& s, u32 f) {
  return (BlockMeta*)s.meta + (a.src_off[f] >> 17) + (a.item_base + f);
}

// unaligned loads built from aligned words (may touch up to 3 bytes past the last byte asked for)
__device__ __forceinline__ u64 ldu64(const u8* p) {
  const u32* w = (const u32*)((uintptr_t)p & ~(uintptr_t)3); const u32 sh = ((u32)(uintptr_t)p & 3) * 8;
  const u32 a0 = w[0], a1 = w[1], a2 = sh ? w[2] : 0;
  return ((u64)__funnelshift_r(a1, a2, sh) << 32) | __funnelshift_r(a0, a1, sh);
}
__device__ __forceinline__ u32 ldu32(const u8* p) {
  const u32* w = (const u32*)((uintptr_t)p & ~(uintptr_t)3); const u32 sh = ((u32)(uintptr_t)p & 3) * 8;
  const u32 a0 = w[0], a1 = sh ? w[1] : 0;
  return __funnelshift_r(a0, a1, sh);
}
// candidate position from a 16-bit table entry: the most recent position below p with those low 16 bits
__device__ __forceinline__ bool cand_from_entry(u32 p, u32 e, u32& cand) {
  u32 d = (p - e) & 0xFFFF; if (d == 0) d = 0x10000;
  cand = p - d;
  return d <= p;
}

// number of equal bytes of src[a..) and src[a-off..), a + n <= end, counted by the whole warp
__device__ __forceinline__ u32 warp_extend(const u8* src, u32 a, u32 off, u32 end, u32 lane) {
  u32 n = 0;
  while (true) {
    const u32 i = a + n + lane;
    const bool eq = i < end && src[i] == src[i - off];
    const unsigned m = __ballot_sync(FULLMASK, eq);
    if (m == FULLMASK) { n += 32; continue; }
    return n + (u32)__ffs(~m) - 1;
  }
}
// the same against a second sequence: number of i >= a with src[i] == ref[i], a + n <= end
__device__ __forceinline__ u32 warp_extend_ref(const u8* src, const u8* ref, u32 a, u32 end, u32 lane) {
  u32 n = 0;
  while (true) {
    const u32 i = a + n + lane;
    const bool eq = i < end && src[i] == ref[i];
    const unsigned m = __ballot_sync(FULLMASK, eq);
    if (m == FULLMASK) { n += 32; continue; }
    return n + (u32)__ffs(~m) - 1;
  }
}

// DICT: the launch compresses with the context's dictionary (EncodeArgs::dict).  Its match tables are looked up by every
// lane whose position found no match in the chunk's own tables, in libzstd's dictMatchState order: chunk long, dictionary
// long, chunk short, dictionary short.  A dictionary match ends at the end of the content, its offset reaches back over
// the chunk into the content, and the first block starts from the dictionary's repeat offsets.
// ACCEL: a negative level, acceleration -a.level (never with DFAST).  The lanes probe libzstd's pairs of adjacent positions
// with a stride of 1 + acceleration (zb_encode.cuh enc_probe_off), so a window covers 16 strides instead of 32 positions.
template <bool DFAST, bool DICT, bool ACCEL>
__global__ void __launch_bounds__(32) k_enc_match(EncodeArgs a, EncodeScratch sc, u32 hlogL, u32 hlogS, u32 mls, u16* gtab) {
  extern __shared__ __align__(16) u16 tabShared[];
  const u32 lane = threadIdx.x, warp = blockIdx.x, nWarps = gridDim.x;
  const EncDict* const ed = DICT ? a.dict : nullptr;
  if (DICT && a.dict_err) return;                               // k_enc_entropy reports it for every item
  const u32* const dtabL = DICT ? enc_dict_table(ed, DFAST ? EDT_LONG : (mls == 6 ? EDT_MLS6 : EDT_MLS5)) : nullptr;
  const u32* const dtabS = DICT ? enc_dict_table(ed, EDT_MLS5) : nullptr;
  const u8* const dc = DICT ? enc_dict_content(ed) : nullptr;
  const u32 dsize = DICT ? ed->contentSize : 0;
  const u32 tw = (1u << hlogL) + (DFAST ? (1u << hlogS) : 0);
  // gtab != nullptr (launches that have the device to themselves): the tables of this warp live in global scratch,
  // kGtabStride bytes per warp, and the launch asks for no shared memory.  This kernel's throughput is its resident warp count (a serial chain per warp with a far
  // memory round trip per sequence), and shared-memory tables bound that at 24 / 12 / 16 warps per SM (levels 1 / 2 / 3) and
  // 9 for chunks above 128 KiB; 32 one-warp CTAs per SM keep 256-384 KB of tables in L1 / L2 instead.  Measured on 1 GiB of
  // log text in 128 KiB chunks: 37.9 -> 28.8 ms (level 1), 60.1 -> 35.4 (level 2), 69.2 -> 50.5 (level 3); tick 1 MiB chunks
  // 198 -> 111 ms.  At equal warp counts the two placements are within 6 % of each other; 40 / 48 / 64 warps per SM
  // (two-warp CTAs, registers capped at 48 / 40 / 32) are slower than 32 on every shape but level-1 log text: the tables no
  // longer stay in L1 (profiles/r2c_enc_match_tables.jsonl).
  u16* const tab = gtab ? gtab + (size_t)warp * (kGtabStride / 2) : tabShared;
  u16* const tabL = tab; u16* const tabS = tab + (1u << hlogL);
  // The unit of work is one BLOCK (<= 128 KiB) of one chunk: blocks of a chunk are matched independently, so a batch of
  // few large chunks spreads over as many warps as a batch of many small ones.  A block that is not the chunk's first
  // starts from a table primed with the ENC_PRIME bytes before it (the positions a table of this size would still
  // remember), and — as before — without repeat offsets.
  const u32 perChunk = a.max_src_size > BLOCKSIZE_MAX ? (a.max_src_size + BLOCKSIZE_MAX - 1) / BLOCKSIZE_MAX : 1;
  for (u64 unit = warp; unit < (u64)a.n * perChunk; unit += nWarps) {
    const u32 f = (u32)(unit / perChunk), blk = (u32)(unit % perChunk), bpos = blk * BLOCKSIZE_MAX;
    const u8* src = a.src_base + a.src_off[f]; const u32 size = a.src_size[f];
    if (blk > 0 && bpos >= size) continue;
    u8* const lits0 = lit_base(a, sc, f); u32* const seqs0 = seq_base(a, sc, f); BlockMeta* const meta = meta_base(a, sc, f);
    for (u32 i = lane; i < tw / 2; i += 32) ((u32*)tab)[i] = 0;
    __syncwarp();
    if (blk > 0) {
      for (u32 q0 = bpos - ENC_PRIME; q0 < bpos; q0 += 32) {
        const u32 q = q0 + lane;
        const u64 v = ldu64(src + q);
        const u32 hL = hash64(v, hlogL, DFAST ? 8 : mls);
        const unsigned mL = __match_any_sync(FULLMASK, hL);
        if ((mL >> lane) == 1) tabL[hL] = (u16)q;                   // the last position of each hash group is the one kept
        if (DFAST) {
          const u32 hS = hash64(v, hlogS, mls);
          const unsigned mS = __match_any_sync(FULLMASK, hS);
          if ((mS >> lane) == 1) tabS[hS] = (u16)q;
        }
        __syncwarp();
      }
    }
    u32 rep1 = DICT ? ed->rep[0] : 1, rep2 = DICT ? ed->rep[1] : 4;   // the decoder starts every frame from the same two
    {
      const u32 bsize = size - bpos < BLOCKSIZE_MAX ? size - bpos : BLOCKSIZE_MAX;
      const u32 bend = bpos + bsize;
      u8* const lits = lits0 + (size_t)blk * BLOCKSIZE_MAX; u32* const seqs = seqs0 + 2 * (size_t)blk * kBlockSeqCap;
      u32 nseq = 0, nlits = 0;
      // all-equal block? (RLE block: the entropy stage handles it, nothing to match)
      bool rle = bsize >= 2;
      if (rle) {
        const u8 b0 = src[bpos];
        for (u32 i0 = bpos; i0 < bend && rle; i0 += 32) { const u32 i = i0 + lane; if (__ballot_sync(FULLMASK, i < bend && src[i] != b0)) rle = false; }
      }
      if (!rle && bsize >= 64) {
        // repeat offsets are only trusted when established inside this block (or the frame's initial 1, 4): an
        // earlier block may end up stored raw, which leaves the decoder's history untouched (DecodeSequence :1576-1596)
        if (blk > 0) { rep1 = 0; rep2 = 0; }
        u32 anchor = bpos; const u32 ilimit = bend - 8;
        u32 p0 = bpos + (bpos == 0 ? 1 : 0);
        // fresh: p0 directly follows a match, so the "immediate repeat of the older offset" test (litLength 0,
        // code 1 == second offset) is pending for it.  Its loads are issued together with the window's, and the
        // window's table lookups and candidate loads run speculatively behind it: one memory round trip instead of two.
        bool fresh = false;
        while (p0 < ilimit || (fresh && p0 == ilimit)) {
          const u32 step = (ACCEL ? 1u - (u32)a.level : 1u) + ((p0 - anchor) >> 8);   // skim incompressible runs
          if (lane < 4) prefetch_line(src + p0 + 384 + 128 * lane);   // the source streams in from HBM: keep ~4 lines ahead in L1
          const u32 p = p0 + enc_probe_off(ACCEL, lane, step);
          const bool act = p < ilimit;
          u32 r2a = 0, r2b = 1;
          if (fresh && rep2 != 0 && (!DICT || rep2 <= p0)) { r2a = ldu32(src + p0); r2b = ldu32(src + p0 - rep2); }   // (without a
                                                                       //  dictionary rep2 is an offset seen in the chunk: always <= p0)
          const u64 v = act ? ldu64(src + p) : 0;
          const u32 hL = act ? hash64(v, hlogL, DFAST ? 8 : mls) : (0x80000000u | lane);
          const u32 eL = act ? tabL[hL] : 0;
          const unsigned mL = __match_any_sync(FULLMASK, hL);
          const unsigned lowL = mL & ((1u << lane) - 1);
          u32 candL; bool validL;
          if (lowL) { candL = p0 + enc_probe_off(ACCEL, 31 - __clz(lowL), step); validL = act; } else validL = cand_from_entry(p, eL, candL) && act;
          u32 hS = 0, candS = 0; bool validS = false; unsigned mS = 0;
          if (DFAST) {
            hS = act ? hash64(v, hlogS, mls) : (0x80000000u | lane);
            const u32 eS = act ? tabS[hS] : 0;
            mS = __match_any_sync(FULLMASK, hS);
            const unsigned lowS = mS & ((1u << lane) - 1);
            if (lowS) { candS = p0 + enc_probe_off(ACCEL, 31 - __clz(lowS), step); validS = act; } else validS = cand_from_entry(p, eS, candS) && act;
          }
          bool okL = false, okS = false;
          if (validL) okL = DFAST ? (ldu64(src + candL) == v) : (ldu32(src + candL) == (u32)v);
          if (DFAST && validS) okS = ldu32(src + candS) == (u32)v;
          u32 candDL = 0, candDS = 0; bool okDL = false, okDS = false;   // dictionary candidates (content positions)
          if (DICT && act && !okL) {
            candDL = dtabL[hash64(v, ENC_DICT_HLOG, DFAST ? 8 : mls)];
            if (candDL != ENC_DICT_EMPTY) okDL = DFAST ? (ldu64(dc + candDL) == v) : (ldu32(dc + candDL) == (u32)v);
          }
          if (DICT && DFAST && act && !okL && !okDL && !okS) {
            candDS = dtabS[hash64(v, ENC_DICT_HLOG, mls)];
            if (candDS != ENC_DICT_EMPTY) okDS = ldu32(dc + candDS) == (u32)v;
          }
          // (ACCEL: the repeat offset is tried at the start of every probe pair but the first, libzstd's ip2)
          const bool rok = act && (!ACCEL || (lane != 0 && !(lane & 1))) && rep1 != 0 && rep1 <= p && ldu32(src + p - rep1) == (u32)v;
          if (fresh) {
            fresh = false;
            if (r2a == r2b) {                                                      // uniform over the warp
              const u32 rlen = 4 + warp_extend(src, p0 + 4, rep2, bend, lane);
              { const u32 t = rep2; rep2 = rep1; rep1 = t; }
              if (lane == 0) {
                tabL[hash64(ldu64(src + p0), hlogL, DFAST ? 8 : mls)] = (u16)p0;
                if (DFAST) tabS[hash64(ldu64(src + p0), hlogS, mls)] = (u16)p0;
                seqs[2 * nseq] = ((rlen - 3) & 0xFFFF) << 16;
                seqs[2 * nseq + 1] = 1u | ((((rlen - 3) >> 16) & 1) << 30);
              }
              __syncwarp();
              nseq++;
              p0 += rlen; anchor = p0;
              fresh = p0 <= ilimit;
              continue;
            }
          }
          const unsigned fRep = __ballot_sync(FULLMASK, rok);
          const unsigned fTab = __ballot_sync(FULLMASK, okL | okS | okDL | okDS);
          const unsigned found = fTab | fRep;
          if (!found) {                                                // no match in the window: enter every position, move on
            if (act && (mL >> lane) == 1) tabL[hL] = (u16)p;          // the last position of each hash group is the one kept
            if (DFAST && act && (mS >> lane) == 1) tabS[hS] = (u16)p;
            __syncwarp();
            p0 += (ACCEL ? 16 : 32) * step; continue;
          }
          u32 fl = (u32)__ffs(found) - 1, probe = 0;
          if (ACCEL) {
            // libzstd's order over the pairs: for pair k the repeat offset at the next pair's start (lane 2k + 2) first, then
            // the table at lane 2k, then at 2k + 1.  probe: where libzstd's current0 is (the fill after the match).
            const unsigned repPair = fRep >> 2;
            const u32 b = (u32)__ffs(repPair | fTab) - 1;
            fl = ((repPair >> b) & 1) ? b + 2 : b;
            probe = p0 + enc_probe_off(true, b, step);
          } else if (!((fRep >> fl) & 1)) {
            // a repeat-offset match up to 3 positions further on beats a table match here (it is cheaper to code)
            const unsigned nearRep = fRep & (0xEu << fl); if (nearRep) fl = (u32)__ffs(nearRep) - 1;
          }
          u32 pos = p0 + enc_probe_off(ACCEL, fl, step);
          // at the winning lane: repeat offset > long/main table > (dictionary long) > short table (> dictionary short)
          const u32 kind = rok ? 0 : (okL ? 1 : (DICT ? (okDL ? 3 : (okS ? 2 : 4)) : 2));
          const u32 kf = __shfl_sync(FULLMASK, kind, fl);
          const u32 cf = __shfl_sync(FULLMASK, DICT ? (kind == 1 ? candL : (kind == 3 ? candDL : (kind == 4 ? candDS : candS))) : (kind == 1 ? candL : candS), fl);
          u32 cnd = kf == 0 ? pos - rep1 : cf;
          const u32 off = (DICT && kf >= 3) ? pos + (dsize - cnd) : pos - cnd;
          // forward extension and backward catch-up (:pos > anchor && cnd > 0 && equal) from one round of loads
          u32 mlen;
          if (DICT && kf >= 3) {
            // against the dictionary (cnd: content position): ref[i] is the byte src[i] is compared with; forward up to the
            // end of the content, backward down to its start or the anchor
            const u8* const ref = dc + cnd - pos;
            const u32 fend = min(bend, pos + (dsize - cnd));
            const u32 i = pos + 4 + lane; const bool feq = i < fend && src[i] == ref[i];
            const u32 maxb = min(pos - anchor, cnd);
            const bool beq = lane < maxb && src[pos - 1 - lane] == ref[pos - 1 - lane];
            const unsigned fm = __ballot_sync(FULLMASK, feq), bm = __ballot_sync(FULLMASK, beq);
            const u32 fwd = fm == FULLMASK ? 32 + warp_extend_ref(src, ref, pos + 36, fend, lane) : (u32)__ffs(~fm) - 1;
            u32 bwd = bm == FULLMASK ? 32 : (u32)__ffs(~bm) - 1;
            if (bm == FULLMASK) while (bwd < maxb && src[pos - 1 - bwd] == ref[pos - 1 - bwd]) bwd++;
            mlen = 4 + fwd + bwd; pos -= bwd;
          } else {
            const u32 i = pos + 4 + lane; const bool feq = i < bend && src[i] == src[i - off];
            const u32 maxb = min(pos - anchor, cnd);
            const bool beq = lane < maxb && src[pos - 1 - lane] == src[cnd - 1 - lane];
            const unsigned fm = __ballot_sync(FULLMASK, feq), bm = __ballot_sync(FULLMASK, beq);
            const u32 fwd = fm == FULLMASK ? 32 + warp_extend(src, pos + 36, off, bend, lane) : (u32)__ffs(~fm) - 1;
            u32 bwd = bm == FULLMASK ? 32 : (u32)__ffs(~bm) - 1;
            if (bm == FULLMASK) while (bwd < maxb && src[pos - 1 - bwd] == src[cnd - 1 - bwd]) bwd++;
            mlen = 4 + fwd + bwd; pos -= bwd; cnd -= bwd;
          }
 {
            // enter the window's positions up to the end of the match: nothing at or beyond the restart position may
            // go in, or it would later be found as its own candidate
            const bool ins = act && p < pos + mlen;
            const unsigned insMask = __ballot_sync(FULLMASK, ins);
            if (ins && ((mL & insMask) >> lane) == 1) tabL[hL] = (u16)p;
            if (DFAST && ins && ((mS & insMask) >> lane) == 1) tabS[hS] = (u16)p;
            __syncwarp();
          }
          const u32 ll = pos - anchor;
          u32 offBase;
          if (kf == 0 && ll > 0) offBase = 1;                          // repeat offset 1; history unchanged
          else { offBase = off + 3; rep2 = rep1; rep1 = off; }         // (a repeat right after a match must be spelled out: with
                                                                       //  litLength 0 the code 1 means the *second* offset, :1511)
          for (u32 i = lane; i < ll; i += 32) lits[nlits + i] = src[anchor + i];
          if (lane == 0) {
            seqs[2 * nseq] = (ll & 0xFFFF) | (((mlen - 3) & 0xFFFF) << 16);
            seqs[2 * nseq + 1] = (offBase & 0x3FFFFFFFu) | ((((mlen - 3) >> 16) & 1) << 30) | (((ll >> 16) & 1) << 31);
          }
          nlits += ll; nseq++;
          anchor = pos + mlen; p0 = anchor;
          if (p0 <= ilimit) {
            if (ACCEL) {              // libzstd's fill: the positions 2 past current0 (probe) and 2 before the match end
              if (lane == 0) { tabL[hash64(ldu64(src + probe + 2), hlogL, mls)] = (u16)(probe + 2); tabL[hash64(ldu64(src + p0 - 2), hlogL, mls)] = (u16)(p0 - 2); }
              __syncwarp();
            }
            fresh = true;                                              // immediate-repeat test at the top of the next pass
          }
        }
        // last literals
        const u32 ll = bend - anchor;
        for (u32 i = lane; i < ll; i += 32) lits[nlits + i] = src[anchor + i];
        nlits += ll;
      }
      if (lane == 0) { meta[blk].nseq = nseq; meta[blk].nlits = nlits; }
    }
  }
}

// DICT: frames name the dictionary (Dictionary_ID field) and a malformed one fails every item
template <bool DICT>
__global__ void __launch_bounds__(128) k_enc_entropy(EncodeArgs a, EncodeScratch sc, u32 slot0, u32 nwarps) {
  __shared__ EntWarp sm[4];
  __shared__ EntLut lut;
  if (threadIdx.x < 36) lut.ll[threadIdx.x] = ll_info(threadIdx.x);
  if (threadIdx.x < 53) lut.ml[threadIdx.x] = ml_info(threadIdx.x);
  __syncthreads();
  const u32 lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const u32 wid = blockIdx.x * 4 + wib;
  if (wid >= nwarps) return;
  EntWarp& w = sm[wib];
  u8* slot = sc.slots + (size_t)(slot0 + wid) * slot_bytes();
  u8* codes = slot; u8* tmp = slot + align16((size_t)kBlockSeqCap * 3);
  for (u32 f = wid; f < a.n; f += nwarps) {
    const u8* src = a.src_base + a.src_off[f]; const u32 size = a.src_size[f];
    u8* dst = a.dst_base + a.dst_off[f]; const u32 cap = a.dst_cap[f];
    u8* const lits0 = lit_base(a, sc, f); u32* const seqs0 = seq_base(a, sc, f); const BlockMeta* meta = meta_base(a, sc, f);
    // frame header (mirror of encode_frame_with)
    const u32 fhs = enc_frame_header_size(size, DICT ? a.dict_id : 0);
    const u32 tail = a.checksum ? 4 : 0;
    u32 res = 0; bool failed = false;
    if (cap < fhs + 3 + tail) { failed = true; res = zerr(ZE_dstSize_tooSmall); }
    if (DICT && a.dict_err) { failed = true; res = zerr(a.dict_err); }
    u32 op = fhs;
    if (!failed && lane == 0) enc_frame_header(dst, size, a.checksum, DICT ? a.dict_id : 0);
    u32 pos = 0, blk = 0;
    if (!failed) do {
      const u32 bsize = size - pos < BLOCKSIZE_MAX ? size - pos : BLOCKSIZE_MAX;
      const u32 last = pos + bsize == size;
      const u8* bstart = src + pos;
      if (op + 3 + tail > cap) { failed = true; res = zerr(ZE_dstSize_tooSmall); break; }
      bool rle = bsize >= 2;
      if (rle) {
        const u8 b0 = bstart[0];
        for (u32 i0 = 0; i0 < bsize && rle; i0 += 32) { const u32 i = i0 + lane; if (__ballot_sync(FULLMASK, i < bsize && bstart[i] != b0)) rle = false; }
      }
      if (rle) {
        if (op + 4 + tail > cap) { failed = true; res = zerr(ZE_dstSize_tooSmall); break; }
        if (lane == 0) { const u32 h = last | (1u << 1) | (bsize << 3); dst[op] = (u8)h; dst[op + 1] = (u8)(h >> 8); dst[op + 2] = (u8)(h >> 16); dst[op + 3] = bstart[0]; }
        op += 4;
      } else {
        u32 csize = 0; bool compressed = false;
        if (bsize >= 64) {
          SeqStore st; st.seqs = seqs0 + 2 * (size_t)blk * kBlockSeqCap; st.n = meta[blk].nseq; st.cap = kBlockSeqCap;
          st.lits = lits0 + (size_t)blk * BLOCKSIZE_MAX; st.nlits = meta[blk].nlits;
          u32 room = bsize - 1 < BLOCKSIZE_MAX - 1 ? bsize - 1 : BLOCKSIZE_MAX - 1;
          const u32 avail = cap - op - 3 - tail;
          if (room > avail) room = avail;
          u8* body = dst + op + 3;
          const EncDict* const edb = DICT && blk == 0 && a.dict->hasEntropy ? a.dict : nullptr;   // (as encode_frame_with)
          const u32 l = warp_enc_literals(body, room, st.lits, st.nlits, w, tmp, lane, edb, a.level < 0);
          if (l) {
            const u32 sq = warp_enc_sequences(body + l, room - l, st, codes, w, lut, a.level, lane, edb);
            if (sq && l + sq < bsize) { csize = l + sq; compressed = true; }
          }
        }
        if (compressed) {
          if (lane == 0) { const u32 h = last | (2u << 1) | (csize << 3); dst[op] = (u8)h; dst[op + 1] = (u8)(h >> 8); dst[op + 2] = (u8)(h >> 16); }
          op += 3 + csize;
        } else {
          if (op + 3 + bsize + tail > cap) { failed = true; res = zerr(ZE_dstSize_tooSmall); break; }
          if (lane == 0) { const u32 h = last | (0u << 1) | (bsize << 3); dst[op] = (u8)h; dst[op + 1] = (u8)(h >> 8); dst[op + 2] = (u8)(h >> 16); }
          op += 3;
          __syncwarp();
          wcopy(dst + op, bstart, bsize, lane);
          op += bsize;
        }
      }
      __syncwarp();
      pos += bsize; blk++;
    } while (pos < size);
    if (lane == 0) a.result[f] = failed ? res : op;
    __syncwarp();
  }
}

__global__ void __launch_bounds__(128) k_enc_xxh(EncodeArgs a) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 f = t >> 2, sub = t & 3, lane = threadIdx.x & 31;
  const unsigned gmask = 0xFu << (lane & ~3u);
  if (f >= a.n) return;
  const u32 r = a.result[f];
  if (is_err(r)) return;
  const u64 h = xxh64_group<false>(a.src_base + a.src_off[f], a.src_size[f], sub, gmask, lane & ~3u);
  if (sub == 0) {
    u8* p = a.dst_base + a.dst_off[f] + r;   // encode_frame_with reserved these 4 bytes
    p[0] = (u8)h; p[1] = (u8)(h >> 8); p[2] = (u8)(h >> 16); p[3] = (u8)(h >> 24);
    a.result[f] = r + 4;
  }
}

EncodeArgs encode_args(const Items& it, size_t n, u32 item_base, int level, int checksum, u32 max_src_size, u32 slot,
                       const void* dict, const std::vector<uint4>* h_dict) {
  EncodeArgs a{};
  a.src_base = it.src; a.src_off = it.srcOff; a.src_size = it.srcSize;
  a.dst_base = it.dst; a.dst_off = it.dstOff; a.dst_cap = it.dstCap; a.result = it.result;
  a.n = (u32)n; a.item_base = item_base; a.level = level; a.checksum = checksum; a.max_src_size = max_src_size; a.stream_slot = slot;
  if (dict) {
    const EncDict* h = reinterpret_cast<const EncDict*>(h_dict->data());
    a.dict = reinterpret_cast<const EncDict*>(dict); a.dict_id = h->dictID; a.dict_err = h->err;
  }
  return a;
}

void dict_load_host(const u8* dict, u32 size, DictState& ds) {
  std::vector<u8> b(dict, dict + size); b.resize((size_t)size + 64, 0);   // the parser may read 64 bytes past the end
  HufBuildWk wk; HufFseScratch fs; u8 slot[260]; s16 norm[64]; u16 next[64];
  dict_load(b.data(), size, ds, wk, fs, slot, norm, next);
}

std::vector<uint4> enc_dict_block(const u8* dict, u32 size, const DictState& ds) {
  std::vector<u8> b(dict, dict + size); b.resize((size_t)size + 64, 0);
  std::vector<uint4> out((enc_dict_bytes(ds.err ? 0 : ds.contentSize) + 15) / 16, uint4{});
  HufBuildWk wk; HufFseScratch fs; u8 slot[260]; std::vector<u8> tableSymbol(512);
  enc_dict_prepare(b.data(), size, ds, reinterpret_cast<EncDict*>(out.data()), wk, fs, slot, tableSymbol.data());
  return out;
}

size_t encode_bound(size_t srcSize) { return srcSize + (srcSize >> 8) + 32 + 3 * ((srcSize >> 17) + 1); }

// Entropy-stage work areas ("slots", one per resident warp).  A launch that owns the context (device-pointer path)
// takes up to kSlotsExclusive from the start of the pool; slices of a host batch that run concurrently on
// different streams each get one of ENC_STREAM_PARTS equal partitions.
static constexpr u32 kPoolSlots = 148 * 16 * 4;
static constexpr u32 kSlotsExclusive = 148 * 24;   // upper bound; the launch uses what is resident (EncodeScratch::entWarps)
static constexpr u32 kSlotsPerPart = kPoolSlots / ENC_STREAM_PARTS;

cudaError_t encode_alloc(EncodeScratch& s, size_t maxBatchBytes, size_t maxItems) {
  s = EncodeScratch();
  s.maxBytes = maxBatchBytes + 16 * maxItems; s.maxItems = maxItems;   // src offsets are 16-byte aligned in the host path
  return cudaSuccess;
}
void encode_free(EncodeScratch& s) {
  if (s.lit) cudaFree(s.lit); if (s.seq) cudaFree(s.seq); if (s.meta) cudaFree(s.meta); if (s.slots) cudaFree(s.slots);
  if (s.gtab) cudaFree(s.gtab);
  s.lit = nullptr; s.seq = nullptr; s.meta = nullptr; s.slots = nullptr; s.gtab = nullptr;
}

static cudaError_t encode_lazy_alloc(EncodeScratch& s) {
  if (s.lit) return cudaSuccess;
  const size_t B = s.maxBytes, N = s.maxItems + 2;
  cudaError_t e;
  if ((e = cudaMalloc(&s.lit, B + 64 * N + 256)) != cudaSuccess ||
      (e = cudaMalloc(&s.seq, (B / 4 + 64 * ((B >> 17) + 1) + 128 * N + 64) * 8)) != cudaSuccess ||
      (e = cudaMalloc(&s.meta, ((B >> 17) + N + 8) * sizeof(BlockMeta))) != cudaSuccess ||
      (e = cudaMalloc(&s.slots, (size_t)kPoolSlots * slot_bytes())) != cudaSuccess) {
    encode_free(s);   // a later call retries from scratch instead of running on a half-built arena
    return e;
  }
  int dev = 0; cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&s.sms, cudaDevAttrMultiProcessorCount, dev);
  // as many entropy-stage warps as are resident at once: every warp then takes the same number of frames (+-1)
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_enc_entropy<false>, 128, 0) != cudaSuccess || nb < 1) nb = 4;
  s.entWarps = (u32)(s.sms * nb * 4);
  if (s.entWarps > kSlotsExclusive) s.entWarps = kSlotsExclusive;
  cudaFuncSetAttribute(k_enc_match<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  cudaFuncSetAttribute(k_enc_match<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  cudaFuncSetAttribute(k_enc_match<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  cudaFuncSetAttribute(k_enc_match<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  cudaFuncSetAttribute(k_enc_match<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  cudaFuncSetAttribute(k_enc_match<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  return cudaSuccess;
}

const char* const kEncodeKernelNames[ENCODE_KERNELS] = {"k_enc_match", "k_enc_entropy", "k_enc_xxh"};

// The match stage of one launch (k_enc_match): table sizes, grid and table placement.  marks: as for encode_launch.
static void match_launch(const EncodeArgs& a, EncodeScratch& s, cudaStream_t st, cudaEvent_t* marks) {
  // match stage: table sizes per level (u16 entries)
  const bool dfast = a.level >= 3, accel = a.level < 0;
  // level 1 and the negative levels: 2^12 (8 KB), level 2: 2^13 (16 KB), level 3: 2^11 long + 2^12 short (12 KB); chunks
  // above 128 KiB: enc_hlog_*.
  // The sizes date from the shared-memory placement (24 / 12 / 16 warps per SM) and are kept: the ratio band is tested
  // with them (lock-step emulation in tests/hostsim: tick records within -2.4 % of libzstd at 128 KiB chunks, log text
  // gains ratio with the smaller tables) and 32 warps' tables still mostly fit L1.
  const bool big = a.max_src_size > BLOCKSIZE_MAX;
  const u32 hlogL = enc_hlog_long(a.level, big), hlogS = enc_hlog_short(a.level, big), mls = enc_mls(a.level);
  const size_t smem = ((size_t)(1u << hlogL) + (dfast ? (1u << hlogS) : 0)) * 2;
  u32 perSm = (u32)((220 * 1024) / (smem + 1024)); if (perSm > 32) perSm = 32;
  const u64 units = (u64)a.n * (a.max_src_size > BLOCKSIZE_MAX ? (a.max_src_size + BLOCKSIZE_MAX - 1) / BLOCKSIZE_MAX : 1);
  u32 grid = (u32)s.sms * perSm; if (grid > units) grid = (u32)units;
  const bool exclusive = a.stream_slot == ENC_EXCLUSIVE;
  // Match tables in global scratch when the launch has the device to itself.  Slices of a host batch run concurrently on
  // several streams, and the entropy stage of one slice then shares SMs with the match stage of another: its 34 KB of shared
  // memory per CTA shrink the L1 the tables would live in (measured: host-path level 1 19.1 -> 16.4 GB/s with global tables),
  // so those launches keep their tables in shared memory.
  u16* gtab = nullptr;
  if (exclusive && smem <= kGtabStride) {
    if (!s.gtab && cudaMalloc(&s.gtab, (size_t)s.sms * kGtabWarpsPerSm * kGtabStride) != cudaSuccess) {
      cudaGetLastError(); s.gtab = nullptr;                      // no room for the 113 MB: this launch keeps shared-memory tables
    }
    if (s.gtab) { gtab = (u16*)s.gtab; grid = (u32)s.sms * kGtabWarpsPerSm; if (grid > units) grid = (u32)units; }
  }
  if (marks) cudaEventRecord(marks[0], st);
  const size_t sm = gtab ? 0 : smem;
  if (a.dict) {
    if (dfast) k_enc_match<true, true, false><<<grid, 32, sm, st>>>(a, s, hlogL, hlogS, mls, gtab);
    else if (accel) k_enc_match<false, true, true><<<grid, 32, sm, st>>>(a, s, hlogL, hlogS, mls, gtab);
    else k_enc_match<false, true, false><<<grid, 32, sm, st>>>(a, s, hlogL, hlogS, mls, gtab);
  } else {
    if (dfast) k_enc_match<true, false, false><<<grid, 32, sm, st>>>(a, s, hlogL, hlogS, mls, gtab);
    else if (accel) k_enc_match<false, false, true><<<grid, 32, sm, st>>>(a, s, hlogL, hlogS, mls, gtab);
    else k_enc_match<false, false, false><<<grid, 32, sm, st>>>(a, s, hlogL, hlogS, mls, gtab);
  }
}

cudaError_t encode_launch(const EncodeArgs& a, EncodeScratch& s, cudaStream_t st, int* launches, cudaEvent_t* marks) {
  if (a.n == 0) return cudaSuccess;
  cudaError_t e = encode_lazy_alloc(s);
  if (e != cudaSuccess) return e;
  match_launch(a, s, st, marks);
  const bool exclusive = a.stream_slot == ENC_EXCLUSIVE;
  const u32 slot0 = exclusive ? 0 : (a.stream_slot % ENC_STREAM_PARTS) * kSlotsPerPart;
  const u32 maxSlots = exclusive ? s.entWarps : kSlotsPerPart;
  const u32 slots = a.n < maxSlots ? a.n : maxSlots;
  if (marks) cudaEventRecord(marks[1], st);
  if (a.dict) k_enc_entropy<true><<<(slots + 3) / 4, 128, 0, st>>>(a, s, slot0, slots);
  else k_enc_entropy<false><<<(slots + 3) / 4, 128, 0, st>>>(a, s, slot0, slots);
  if (marks) cudaEventRecord(marks[2], st);
  if (launches) *launches += 2;
  if (a.checksum) { k_enc_xxh<<<(a.n * 4 + 127) / 128, 128, 0, st>>>(a); if (launches) *launches += 1; }
  if (marks) cudaEventRecord(marks[3], st);
  return cudaGetLastError();
}

// ---- statistics of the match stage (dictionary training, zb_dict_train.cuh) ----------------------------------------------
// One warp per item, first block only: its literal bytes and the LL / ML / OF codes of its sequences, counted in shared memory
// and added to st[0..DT_STAT_WORDS) (lit[256], ll[36], ml[53], of[32]: the layout of DtStats).
__global__ void __launch_bounds__(256) k_enc_stats(EncodeArgs a, EncodeScratch sc, u32* st) {
  __shared__ u32 h[DT_STAT_WORDS];
  for (u32 i = threadIdx.x; i < DT_STAT_WORDS; i += blockDim.x) h[i] = 0;
  __syncthreads();
  u32* const hl = h; u32* const hll = h + 256; u32* const hml = hll + MaxLL + 1; u32* const hof = hml + MaxML + 1;
  const u32 lane = threadIdx.x & 31, nw = gridDim.x * (blockDim.x >> 5);
  for (u32 f = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); f < a.n; f += nw) {
    const BlockMeta m = meta_base(a, sc, f)[0];
    const u8* lits = lit_base(a, sc, f);
    for (u32 i = lane; i < m.nlits; i += 32) atomicAdd(&hl[lits[i]], 1u);
    SeqStore q; q.seqs = seq_base(a, sc, f); q.n = m.nseq; q.cap = kBlockSeqCap; q.lits = nullptr; q.nlits = 0;
    for (u32 i = lane; i < m.nseq; i += 32) {
      u32 ll, ob, mlm3; seq_get(q, i, ll, ob, mlm3);
      atomicAdd(&hll[ll_code(ll)], 1u); atomicAdd(&hml[ml_code(mlm3)], 1u); atomicAdd(&hof[highbit(ob)], 1u);
    }
  }
  __syncthreads();
  for (u32 i = threadIdx.x; i < DT_STAT_WORDS; i += blockDim.x) if (h[i]) atomicAdd(&st[i], h[i]);
}

cudaError_t encode_match_stats(const EncodeArgs& a, EncodeScratch& s, cudaStream_t st, u32* stats, int* launches) {
  if (a.n == 0) return cudaSuccess;
  if (a.max_src_size > BLOCKSIZE_MAX || !a.dict) return cudaErrorInvalidValue;
  cudaError_t e = encode_lazy_alloc(s);
  if (e != cudaSuccess) return e;
  match_launch(a, s, st, nullptr);
  u32 grid = (a.n + 7) / 8; if (grid > (u32)s.sms * 8) grid = (u32)s.sms * 8;
  k_enc_stats<<<grid, 256, 0, st>>>(a, s, stats);
  if (launches) *launches += 2;
  return cudaGetLastError();
}

}  // namespace zb
