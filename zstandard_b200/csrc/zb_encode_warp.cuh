// zb_encode_warp.cuh — the warp-parallel section writers of k_enc_entropy (encode_kernels.cu): the literals section
// (warp_enc_literals) and the sequences section (warp_enc_sequences) of one block, one warp per call.  Kept in a header
// so that a test harness can drive them directly with crafted sequence stores (tests/gpu_harness/enc_sections.cu).
#pragma once
#include "zb_encode.cuh"

namespace zb {

#define FULLMASK 0xFFFFFFFFu
static constexpr u32 kBlockSeqCap = BLOCKSIZE_MAX / 4 + 64;

__host__ __device__ inline size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }
static constexpr u32 kStreamTmp = 48 * 1024;   // worst case of one Huffman stream: 32 Ki symbols x 11 bits
__host__ __device__ inline size_t slot_bytes() { return align16((size_t)kBlockSeqCap * 3) + 4 * (size_t)kStreamTmp; }

// ---- entropy stage, one warp per frame -------------------------------------------------------------
// Same decisions and same bytes as enc_literals / enc_sequences / encode_frame_with in zb_encode.cuh (the
// serial replay), with the data-parallel parts spread over the lanes: histograms (shared-memory atomics),
// the four Huffman streams (one lane each, into scratch, then concatenated), code computation, block copies.
// Table construction (Huffman tree, FSE normalisation) stays on lane 0.
struct __align__(16) EntWarp {
  u32 hist[256];
  HufEnc he;
  union {                        // the Huffman tree is built before any of the sequence tables exist
    struct { u32 cnt[3][64]; u16 state[3][514 + 2]; u8 sym[512 + 16]; };
    HufBuildScratch hb;
  };
  FseCTable ct[3];
};

__device__ __forceinline__ void wcopy(u8* dst, const u8* src, u32 n, u32 lane) {
  if (n >= 64 && ((((uintptr_t)dst) ^ ((uintptr_t)src)) & 15) == 0) {
    const u32 head = (u32)(-(intptr_t)dst) & 15;
    if (lane < head) dst[lane] = src[lane];
    const u32 body = (n - head) & ~15u;
    const uint4* s4 = (const uint4*)(src + head); uint4* d4 = (uint4*)(dst + head);
    for (u32 i = lane; i < body / 16; i += 32) d4[i] = s4[i];
    for (u32 i = head + body + lane; i < n; i += 32) dst[i] = src[i];
    return;
  }
  for (u32 i = lane; i < n; i += 32) dst[i] = src[i];
}
__device__ __forceinline__ u32 warp_scan_incl(u32 v, u32 lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const u32 t = __shfl_up_sync(FULLMASK, v, d); if (lane >= (u32)d) v += t; }
  return v;
}
struct EntLut { u32 ll[36], ml[53]; };   // per code: base | extra-bit count << 24 (ll_info / ml_info), shared by the CTA's warps
__device__ __forceinline__ u32 wmax(u32 v) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) { const u32 t = __shfl_xor_sync(FULLMASK, v, d); v = t > v ? t : v; }
  return v;
}

// literals section; returns bytes written, 0 = no room (mirror of enc_literals; ed likewise: the dictionary for the first block).
// rawOnly (the negative levels): always raw, as libzstd's fast strategy with a non-zero targetLength
__device__ u32 warp_enc_literals(u8* out, u32 cap, const u8* lits, u32 n, EntWarp& w, u8* tmp, u32 lane, const EncDict* ed, bool rawOnly) {
  const u32 rawLh = n < 32 ? 1 : (n < 4096 ? 2 : 3);
  auto raw = [&]() -> u32 {
    if (rawLh + n > cap) return 0;
    if (lane == 0) {
      if (rawLh == 1) out[0] = (u8)(n << 3); else if (rawLh == 2) { const u32 v = (1u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); }
      else { const u32 v = (3u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); }
    }
    wcopy(out + rawLh, lits, n, lane);
    __syncwarp();
    return rawLh + n;
  };
  if (n < 64 || rawOnly) return raw();
  for (u32 i = lane; i < 256; i += 32) w.hist[i] = 0;
  __syncwarp();
  for (u32 i = lane; i < n; i += 32) atomicAdd(&w.hist[lits[i]], 1u);
  __syncwarp();
  u32 myMaxSym = 0, myLargest = 0;
  for (u32 sI = lane; sI < 256; sI += 32) { const u32 c = w.hist[sI]; if (c) myMaxSym = sI; if (c > myLargest) myLargest = c; }
  const u32 maxSym = wmax(myMaxSym), largest = wmax(myLargest);
  if (largest == n) {
    if (rawLh + 1 > cap) return 0;
    if (lane == 0) {
      if (rawLh == 1) out[0] = (u8)(1 | (n << 3)); else if (rawLh == 2) { const u32 v = 1 | (1u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); }
      else { const u32 v = 1 | (3u << 2) | (n << 4); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); }
      out[rawLh] = lits[0];
    }
    __syncwarp();
    return rawLh + 1;
  }
  if (largest <= (n >> 7) + 4) return raw();
  u32 maxBits = fse_optimal_log(11, n, maxSym, 1); if (maxBits > 11) maxBits = 11;
  // sort the used symbols by (count, symbol) across the warp: rank = number of used symbols that sort before
  // (same order as huf_sort_symbols' stable insertion sort), then lane 0 builds the tree from shared memory
  // keys count << 8 | symbol are distinct and order exactly as the insertion sort does; unused symbols get the
  // largest key.  Every lane ranks its 8 symbols against all 256 keys, read four at a time.
  u32* const keys = reinterpret_cast<u32*>(&w.he);              // 1 KB, free until the code is built
  u32 myKey[8];
#pragma unroll
  for (int k = 0; k < 8; k++) { const u32 s = 32 * k + lane, c = w.hist[s]; myKey[k] = c ? (c << 8) | s : 0xFFFFFFFFu; keys[s] = myKey[k]; }
  __syncwarp();
  u32 rank[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (u32 t = 0; t < 256; t += 4) {
    const uint4 q = *reinterpret_cast<const uint4*>(keys + t);
#pragma unroll
    for (int k = 0; k < 8; k++) rank[k] += (q.x < myKey[k]) + (q.y < myKey[k]) + (q.z < myKey[k]) + (q.w < myKey[k]);
  }
  u32 nUsed = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const bool used = myKey[k] != 0xFFFFFFFFu;
    nUsed += __popc(__ballot_sync(FULLMASK, used));
    if (used) w.hb.order[rank[k]] = (u16)(32 * k + lane);
  }
  __syncwarp();
  u32 ok = 0;
  if (lane == 0) ok = huf_build_sorted(w.he, w.hist, nUsed, maxBits, w.hb) ? 1 : 0;
  ok = __shfl_sync(FULLMASK, ok, 0);
  if (!ok) return raw();
  const bool single = n < 256;
  const u32 lhSize = 3 + (n >= 1024) + (n >= 16384);
  if (lhSize + 8 > cap) return 0;
  u8* body = out + lhSize; const u32 bodyCap = cap - lhSize;
  u32 hdr = 0;
  if (lane == 0) hdr = huf_write_header(body, bodyCap, w.he, w.state[0], w.sym);
  hdr = __shfl_sync(FULLMASK, hdr, 0);
  if (!hdr) return raw();
  __syncwarp();
  u32 tl = 0;
  if (ed && lane == 0) tl = huf_dict_better(ed->huf, w.he, hdr, w.hist) ? 1 : 0;
  const bool treeless = ed && __shfl_sync(FULLMASK, tl, 0);
  const HufEnc& code = treeless ? ed->huf : w.he;             // the dictionary's code is read from global memory, through L1
  u32 csize = treeless ? 0 : hdr;
  if (single) {
    u32 sz = 0;
    if (lane == 0) sz = huf_encode_stream(body + csize, bodyCap - csize, lits, n, code);
    sz = __shfl_sync(FULLMASK, sz, 0);
    if (!sz) return raw();
    csize += sz;
  } else {
    const u32 seg = (n + 3) / 4;
    if (csize + 6 > bodyCap) return raw();
    u32 sz = 0;
    if (lane < 4) { const u32 from = lane * seg, len = lane < 3 ? seg : n - 3 * seg; sz = huf_encode_stream(tmp + (size_t)lane * kStreamTmp, kStreamTmp, lits + from, len, code); }
    const u32 s0 = __shfl_sync(FULLMASK, sz, 0), s1 = __shfl_sync(FULLMASK, sz, 1), s2 = __shfl_sync(FULLMASK, sz, 2), s3 = __shfl_sync(FULLMASK, sz, 3);
    if (!s0 || !s1 || !s2 || !s3 || s0 > 65535 || s1 > 65535 || s2 > 65535 || s3 > 65535) return raw();
    if (csize + 6 + s0 + s1 + s2 + s3 > bodyCap) return raw();
    if (lane == 0) { u8* j = body + csize; j[0] = (u8)s0; j[1] = (u8)(s0 >> 8); j[2] = (u8)s1; j[3] = (u8)(s1 >> 8); j[4] = (u8)s2; j[5] = (u8)(s2 >> 8); }
    csize += 6;
    __syncwarp();
    wcopy(body + csize, tmp, s0, lane); csize += s0;
    wcopy(body + csize, tmp + kStreamTmp, s1, lane); csize += s1;
    wcopy(body + csize, tmp + 2 * (size_t)kStreamTmp, s2, lane); csize += s2;
    wcopy(body + csize, tmp + 3 * (size_t)kStreamTmp, s3, lane); csize += s3;
  }
  const u32 minGain = (n >> 6) + 2;
  if (csize + minGain >= n) return raw();
  if (lane == 0) {
    const u32 lt = treeless ? 3 : 2;
    if (lhSize == 3) { const u32 v = lt | ((single ? 0u : 1u) << 2) | (n << 4) | (csize << 14); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); }
    else if (lhSize == 4) { const u32 v = lt | (2u << 2) | (n << 4) | (csize << 18); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); out[3] = (u8)(v >> 24); }
    else { const u32 v = lt | (3u << 2) | (n << 4) | (csize << 22); out[0] = (u8)v; out[1] = (u8)(v >> 8); out[2] = (u8)(v >> 16); out[3] = (u8)(v >> 24); out[4] = (u8)(csize >> 10); }
  }
  __syncwarp();
  return lhSize + csize;
}

// sequences section; returns bytes written, 0 on failure (mirror of enc_sequences; a repeat-mode table of the dictionary is
// copied into w.ct with its state table left in global memory)
__device__ u32 warp_enc_sequences(u8* out, u32 cap, const SeqStore& st, u8* codes, EntWarp& w, const EntLut& lut, int level, u32 lane,
                                  const EncDict* ed) {
  const u32 nbSeq = st.n;
  if (cap < 4) return 0;
  u32 op = 0;
  if (lane == 0) op = enc_seq_count_header(out, nbSeq);
  op = __shfl_sync(FULLMASK, op, 0);
  if (nbSeq == 0) { __syncwarp(); return op; }
  u8 *llc = codes, *ofc = codes + st.cap, *mlc = codes + 2 * st.cap;
  for (u32 i = lane; i < 3 * 64; i += 32) (&w.cnt[0][0])[i] = 0;
  __syncwarp();
  for (u32 i = lane; i < nbSeq; i += 32) {
    u32 ll, ob, mlm3; seq_get(st, i, ll, ob, mlm3);
    const u32 lc = ll_code(ll), oc = highbit(ob), mc = ml_code(mlm3);
    llc[i] = (u8)lc; ofc[i] = (u8)oc; mlc[i] = (u8)mc;
    atomicAdd(&w.cnt[KIND_LL][lc], 1u); atomicAdd(&w.cnt[KIND_OF][oc], 1u); atomicAdd(&w.cnt[KIND_ML][mc], 1u);
  }
  __syncwarp();
  u32 total = 0, o2w = 0;
  if (lane == 0) {
    bool good = true; u32 used, o2 = op;
    u8* modeByte = out + o2++;
    const SeqKind kLL = seq_kind(KIND_LL), kOF = seq_kind(KIND_OF), kML = seq_kind(KIND_ML);
    u32 mLL = 0, mOF = 0, mML = 0;
    mLL = enc_seq_table_counts_dict(w.ct[0], w.state[0], w.sym, w.cnt[KIND_LL], llc[nbSeq - 1], nbSeq, kLL, level, out + o2, cap - o2, &used, ed, KIND_LL);
    if (mLL == 0xFF) good = false; else o2 += used;
    if (good) { mOF = enc_seq_table_counts_dict(w.ct[1], w.state[1], w.sym, w.cnt[KIND_OF], ofc[nbSeq - 1], nbSeq, kOF, level, out + o2, cap - o2, &used, ed, KIND_OF); if (mOF == 0xFF) good = false; else o2 += used; }
    if (good) { mML = enc_seq_table_counts_dict(w.ct[2], w.state[2], w.sym, w.cnt[KIND_ML], mlc[nbSeq - 1], nbSeq, kML, level, out + o2, cap - o2, &used, ed, KIND_ML); if (mML == 0xFF) good = false; else o2 += used; }
    if (good) { *modeByte = (u8)((mLL << 6) | (mOF << 4) | (mML << 2)); o2w = o2; }
  }
  o2w = __shfl_sync(FULLMASK, o2w, 0);
  if (o2w) {
    // ---- bitstream (mirror of enc_seq_bitstream: same bits, found in parallel) ----
    // The three FSE state chains are serial, but independent of each other and of the bit positions: lanes 0-2 walk
    // them for a chunk of kChunk sequences (last to first) and leave each sequence's state bits in shared memory.
    // All lanes then size their sequences' six fields, a warp prefix sum gives every field its bit offset, and the
    // fields are OR-ed into a shared-memory bit buffer that is flushed to the frame in whole aligned words.
    constexpr u32 kChunk = 64, kBufWords = 184;   // a sequence is <= 88 bits: 64 * 88 + 31 carried bits < 184 * 32
    static_assert(sizeof(w.hist) >= kChunk * 16 && sizeof(w.he) >= (kChunk + kBufWords) * 4, "chunk buffers");
    u32* const sq = w.hist;                                     // [2 * kChunk] the chunk's sequences, write order
    u32* const sbLL = w.hist + 2 * kChunk; u32* const sbML = w.hist + 3 * kChunk;
    u32* const sbOF = reinterpret_cast<u32*>(&w.he);           // code, later state bits | nbBits << 16 | code << 24
    u32* const bitbuf = sbOF + kChunk;
    u8* const s0 = out + o2w;
    u32* const gbase = reinterpret_cast<u32*>((uintptr_t)s0 & ~(uintptr_t)3);
    u32 G = 8 * (u32)((uintptr_t)s0 & 3);                       // stream bit position relative to gbase
    const u32 capBits = 8 * (u32)((out + cap) - reinterpret_cast<u8*>(gbase));
    u32 carry = 0;
    if (G) { if (lane == 0) carry = gbase[0] & ((1u << G) - 1); carry = __shfl_sync(FULLMASK, carry, 0); }   // bytes before the stream ride along
    const FseCTable& myCt = w.ct[lane == 0 ? 0 : (lane == 1 ? 2 : 1)];   // lane 0: LL, 1: ML, 2: OF
    u32* const mySb = lane == 0 ? sbLL : (lane == 1 ? sbML : sbOF);
    u32 state = 0; bool fits = true;
    for (u32 hi = nbSeq; hi > 0 && fits;) {
      const u32 lo = hi > kChunk ? hi - kChunk : 0, cnt = hi - lo;
      __syncwarp();
      for (u32 t = lane; t < cnt; t += 32) {                   // t-th sequence written = sequence hi - 1 - t
        const u32 n = hi - 1 - t;
        const uint2 s2 = *reinterpret_cast<const uint2*>(st.seqs + 2 * (size_t)n);
        sq[2 * t] = s2.x; sq[2 * t + 1] = s2.y;
        sbLL[t] = llc[n]; sbML[t] = mlc[n]; sbOF[t] = ofc[n];
      }
      for (u32 i = lane; i < kBufWords; i += 32) bitbuf[i] = i == 0 ? carry : 0;
      __syncwarp();
      if (lane < 3) {
        for (u32 t = 0; t < cnt; t++) {
          const u32 code = mySb[t];
          if (hi == nbSeq && t == 0) { fse_init_state(myCt, state, code); mySb[t] = code << 24; }   // the first symbol costs no bits
          else {
            const u32 nb = (state + myCt.deltaNbBits[code]) >> 16;                                  // fse_encode
            mySb[t] = (state & ((1u << nb) - 1)) | (nb << 16) | (code << 24);
            state = myCt.stateTable[(i32)(state >> nb) + myCt.deltaFindState[code]];
          }
        }
      }
      __syncwarp();
      u32 run = G & 31;
      for (u32 t0 = 0; t0 < cnt; t0 += 32) {
        const u32 t = t0 + lane; const bool valid = t < cnt;
        u32 fv[6], fn[6], len = 0;
        if (valid) {
          const u32 a = sq[2 * t], bb = sq[2 * t + 1], eLL = sbLL[t], eML = sbML[t], eOF = sbOF[t];
          const u32 ll = (a & 0xFFFF) | ((bb >> 31) << 16), mlm3 = (a >> 16) | (((bb >> 30) & 1) << 16), ob = bb & 0x3FFFFFFFu;   // seq_get
          const u32 lc = eLL >> 24, mc = eML >> 24, oc = eOF >> 24;
          const u32 iLL = lut.ll[lc], iML = lut.ml[mc];
          fv[0] = eOF & 0xFFFF; fn[0] = (eOF >> 16) & 0xFF;    // write order: OF, ML, LL state bits, then litLength,
          fv[1] = eML & 0xFFFF; fn[1] = (eML >> 16) & 0xFF;    // matchLength and offset extra bits
          fv[2] = eLL & 0xFFFF; fn[2] = (eLL >> 16) & 0xFF;
          fv[3] = ll - (iLL & 0xFFFFFF); fn[3] = iLL >> 24;
          fv[4] = mlm3 + 3 - (iML & 0xFFFFFF); fn[4] = iML >> 24;
          fv[5] = ob - (1u << oc); fn[5] = oc;
#pragma unroll
          for (int k = 0; k < 6; k++) len += fn[k];
        }
        const u32 incl = warp_scan_incl(len, lane);
        u32 pos = run + incl - len;
        if (valid) {
#pragma unroll
          for (int k = 0; k < 6; k++) {
            if (fn[k]) {
              const u32 wi = pos >> 5, sh = pos & 31;
              atomicOr(&bitbuf[wi], fv[k] << sh);
              if (sh + fn[k] > 32) atomicOr(&bitbuf[wi + 1], fv[k] >> (32 - sh));
              pos += fn[k];
            }
          }
        }
        run += __shfl_sync(FULLMASK, incl, 31);
      }
      __syncwarp();
      const u32 words = run >> 5, wordBase = G >> 5;
      if ((G & ~31u) + run + 1 > capBits) { fits = false; break; }   // (+ the end mark) out of room: the caller stores the block raw
      for (u32 i = lane; i < words; i += 32) gbase[wordBase + i] = bitbuf[i];
      carry = bitbuf[words];                                        // the incomplete word, if any, leads the next chunk
      G = (G & ~31u) + run;
      hi = lo;
    }
    // state flush (ML, OF, LL) and end mark by lane 0, continuing from the carried bits
    const u32 sLL = __shfl_sync(FULLMASK, state, 0), sML = __shfl_sync(FULLMASK, state, 1), sOF = __shfl_sync(FULLMASK, state, 2);
    __syncwarp();
    if (fits && lane == 0) {
      BitWriter bw; bw.p = reinterpret_cast<u8*>(gbase + (G >> 5)); bw.end = out + cap; bw.acc = carry; bw.nb = G & 31; bw.ovf = false;
      fse_flush_state(bw, w.ct[2], sML); fse_flush_state(bw, w.ct[1], sOF); fse_flush_state(bw, w.ct[0], sLL);
      u8* e = bw_close(bw);
      if (e) total = (u32)(e - out);
    }
  }
  total = __shfl_sync(FULLMASK, total, 0);
  __syncwarp();
  return total;
}

}  // namespace zb
