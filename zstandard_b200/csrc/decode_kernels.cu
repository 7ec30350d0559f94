// decode_kernels.cu — sm_100a kernels of the batched zstd frame decoder.
//
// Pipeline per batch (all on one stream unless the host overlaps sub-batches):
//   k_parse : thread / item     frame header, skippable frames, early verdicts      (ZStdDecompress.cs:2096-2160, 389-499)
//   k_huf   : 4 lanes / frame   Huffman literals -> literal scratch                  (HufDecompress.cs:117-358)
//   k_seq   : thread / frame    FSE tables + sequence bitstream -> 8-byte records    (ZStdDecompress.cs:958-1180, 1443-1608)
//   k_exec  : warp / frame      literal copy + match copy into dst, raw/RLE blocks   (ZStdDecompress.cs:1212-1352, 1599-1605, 2033-2091)
//   k_xxh   : 4 lanes / frame   XXH64 content checksum                               (XxHash.cs:896-1161)
#include "zb_decode.cuh"
#include "decode_kernels.cuh"
#include "xxh_device.cuh"
#ifdef ZB_EXEC_DEBUG
#include <stdio.h>
#endif

namespace zb {

// -----------------------------------------------------------------------------------------------
// scratch addressing shared by the stages (see DESIGN.md "HBM layout")
// -----------------------------------------------------------------------------------------------
// A data frame of item f writes at dst_off[f] + out_base and may use dst_cap[f] - out_base bytes (out_base > 0 only
// for the second and later data frames of one item); its scratch regions follow from that position, so they stay
// inside the item's share of the arenas.
__device__ __forceinline__ u64 frame_dst_off(const DecodeArgs& a, u32 f, const FrameInfo& fi) { return a.dst_off[f] + fi.out_base; }
__device__ __forceinline__ u32 frame_cap(const DecodeArgs& a, u32 f, const FrameInfo& fi) { return a.dst_cap[f] - fi.out_base; }
__device__ __forceinline__ u8* lit_region(const DecodeArgs& a, u32 f, const FrameInfo& fi) { return a.lit_arena + (frame_dst_off(a, f, fi) & ~15ull) + 64ull * (a.item_base + f); }
__device__ __forceinline__ u64 lit_capacity(u32 cap) { return (u64)cap + 40; }
__device__ __forceinline__ SeqRec* seq_region(const DecodeArgs& a, u32 f, const FrameInfo& fi) { return a.seq_arena + 2 * (frame_dst_off(a, f, fi) / 3) + 32ull * (a.item_base + f); }

// first unit of this launch's range of the unit arena: a frame may list cap / PAR_UNIT_BYTES + PAR_UNIT_SLACK units, so the
// ranges of the slices that share the arena follow from dst_off / item_base like the other scratch regions and cannot meet
__device__ __forceinline__ u64 unit_slice_base(const DecodeArgs& a) { return a.dst_off[0] / PAR_UNIT_BYTES + (u64)PAR_UNIT_SLACK * a.item_base; }

// =================================================================================================
// k_parse
// =================================================================================================
// one item: parse, early verdicts, BlockUnits of multi-block frames.  Returns the sequence-kernel list the item's frame is
// entered in (0 = FI_SEQ_A, 1 = FI_SEQ_B, 2 = full-size tables), -1 = none (finished here, or block-parallel)
__device__ __forceinline__ int parse_one(const DecodeArgs& a, u32 i) {
  FrameInfo fi; u32 r = 0; u32 start = 0, outBase = 0;
  if (a.pass) {
    // later passes only touch items whose previous data frame decoded cleanly and is followed by another one
    const FrameInfo prev = a.info[i];
    if ((prev.flags & FI_DONE) || prev.next_off == 0 || is_err(a.result[i])) { a.info[i].flags = FI_DONE; return -1; }
    start = prev.next_off; outBase = prev.out_base + prev.decoded;
  }
  const u8* src = a.src_base + a.src_off[i];
  bool go = parse_item(src, a.src_size[i], fi, &r, start, outBase, a.dict ? a.dict->err : 0, a.dict ? a.dict->dictID : 0);
  if (go && a.units) {
    // multi-block frames whose structure is sound become BlockUnits (zb_blocks.cuh): count, reserve, fill
    const u32 cap = a.dst_cap[i] - fi.out_base, maxU = cap / PAR_UNIT_BYTES + PAR_UNIT_SLACK;
    const u32 nu = par_walk(src, a.src_size[i], fi.body_off, lit_capacity(cap), seq_capacity(cap), a.dict, maxU, nullptr, i);
    if (nu) {
      const u32 base = atomicAdd(a.cnt, nu);
      par_walk(src, a.src_size[i], fi.body_off, lit_capacity(cap), seq_capacity(cap), a.dict, maxU, a.units + unit_slice_base(a) + base, i);
      fi.flags |= FI_PAR; fi.unit_base = base; fi.unit_count = nu;
      a.par_list[a.item_base + atomicAdd(a.cnt + 1, 1u)] = i;
    }
  }
  int list = -1;
  if (go) {
    // frames of few literals go to the Huffman kernel with the small root table (k_huf<HUF_ROOT_SMALL>), frames of few
    // sequences to a sequence kernel with small tables (a dictionary's tables are full size): zb_format.cuh
    bool fewLiterals;
    u32 cls = first_block_classes(src + fi.body_off, a.src_size[i] - fi.body_off, a.seq_a_max, a.seq_b_max, &fewLiterals);
    if (fewLiterals) { fi.flags |= FI_SMALLHUF; atomicAdd(a.cnt + 2, 1u); }
    if (a.dict && a.dict->hasEntropy) cls = 0;
    if (!(fi.flags & FI_PAR)) {
      if (cls == 1) fi.flags |= FI_SEQ_A; else if (cls == 2) fi.flags |= FI_SEQ_B;
      list = cls == 0 ? 2 : (int)cls - 1;                                           // lists / counters in the order A, B, full size
    }
  }
  a.info[i] = fi;
  if (!go) a.result[i] = r;
  return list;
}

__global__ void __launch_bounds__(128) k_parse(DecodeArgs a) {
  __shared__ u32 warpCount[3][4], ctaBase[3];
  const u32 i = blockIdx.x * 128 + threadIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int list = i < a.n ? parse_one(a, i) : -1;
  // Every frame of the frame-serial path is entered in its class's dense list (the sequence kernels take 32 consecutive
  // entries per warp, so a launch of mixed classes wastes no lanes).  The lists keep the items' order inside a CTA's 128
  // items (ranks from ballots, one reservation per CTA and list): the 32 frames of a sequence-kernel warp stay neighbours
  // in the source / record arenas.  (Appending item by item scrambles the lists over the whole batch, which cost the
  // sequence kernel 22-29 % on every shape measured: 1.69 -> 2.06 ms on the 64 KiB log frames.)
  u32 rank = 0;
  for (int k = 0; k < 3; k++) {
    const unsigned m = __ballot_sync(0xFFFFFFFFu, list == k);
    if (list == k) rank = __popc(m & ((1u << lane) - 1));
    if (lane == 0) warpCount[k][w] = __popc(m);
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const u32 t = warpCount[threadIdx.x][0] + warpCount[threadIdx.x][1] + warpCount[threadIdx.x][2] + warpCount[threadIdx.x][3];
    ctaBase[threadIdx.x] = t ? atomicAdd(a.cnt + 3 + threadIdx.x, t) : 0;
  }
  __syncthreads();
  if (list >= 0) {
    u32 before = 0;
    for (u32 j = 0; j < w; j++) before += warpCount[list][j];
    a.par_list[(size_t)(1 + list) * a.list_stride + a.item_base + ctaBase[list] + before + rank] = i;
  }
}

// =================================================================================================
// k_huf : one warp per CTA, 8 frames per warp, lanes 4f..4f+3 own the 4 streams of frame f
// =================================================================================================
// The kernel is bound by how many frames an SM holds (one warp decodes eight frames' streams as eight dependent lookup
// chains).  What it keeps in shared memory is a ROOT table of 2^R cells (zb_format.cuh huf_fill_root); codes longer than R
// bits are looked up in the full table, which lives in a per-CTA-slot region of global memory (DecodeArgs::huf_full; only
// the long codes' cells are ever written or read there).  Two instantiations share the frames: R = 9 (1 KB per frame,
// 11 CTAs per SM) takes the frames k_parse marked FI_SMALLHUF — at most 2 048 literals in their first block, for which every
// known encoder chooses a table log <= 9, so nothing is ever "long" (a crafted frame that is takes the long path and is
// still decoded correctly) — and R = 11 (4 KB per frame, 5 CTAs per SM) the others, where only the 12-bit codes of a log-12
// table are long.  (Measured: R = 9 for every frame costs 2.7 ms instead of 1.2 ms on 64 KiB tick frames, whose 256-symbol
// alphabets put a quarter of the symbols on 10- and 11-bit codes; on 4 KiB frames it is 2.8 ms against 4.7 ms.)
template <int R> struct HufSmem {
  __align__(16) u16 root[8][1 << R];               // while a frame's weights are read, its cells hold the weights' FSE cells
  HufBuildWk wk[8];
  __align__(16) u32 ring[32][ZB_RING_WORDS + 4];   // per-lane (= per-stream) bitstream read-ahead (BitRing).  While a frame's
                                                   // weights are read, the group's four rings hold norm / symbolNext of the
                                                   // weights' FSE table, then the second ring the per-symbol slots
};
static_assert(4 * (ZB_RING_WORDS + 4) * 4 >= 1024 && (sizeof(u16) << HUF_ROOT_SMALL) >= 256, "FSE scratch of the weights must fit");
// full table of one resident frame: 2^11 cells + the 256-byte side table of a folded log-12 table
#define HUF_FULL_STRIDE ((1u << HUF_TABLE_LOG) + 128u)   // in u16
size_t decode_huf_full_bytes(int ctas) { return (size_t)ctas * 8 * HUF_FULL_STRIDE * sizeof(u16); }


// weights at (tb, tbSize) -> root table in shared memory (+ the long codes in the slot's full table); group-uniform result
template <int R>
__device__ __forceinline__ bool huf_build_tables(HufSmem<R>& sm, u32 slot, u32 sub, unsigned gmask, const u8* tb, u32 tbSize, u16* fullMem,
                                                 HufTabs& T, u32* hdrOut) {
  HufBuildWk& wk = sm.wk[slot];
  u8* const slotMem = (u8*)&sm.ring[slot * 4 + 1][0];
  u32 hdr = 0, nbSym = 0, tl = 0, e = 0;
  if (sub == 0) {
    HufFseScratchRef fs{(s16*)&sm.ring[slot * 4][0], (u16*)((u8*)&sm.ring[slot * 4][0] + 512), (u32*)sm.root[slot]};
    e = huf_read_weights(tb, tbSize, wk, fs, slotMem, &hdr, &tl, &nbSym);
    if (!e && hdr >= tbSize) e = ZE_srcSize_wrong;                                 // HufDecompress.cs:1193
  }
  __syncwarp(gmask);
  e = __shfl_sync(gmask, e, slot * 4); hdr = __shfl_sync(gmask, hdr, slot * 4);
  tl = __shfl_sync(gmask, tl, slot * 4); nbSym = __shfl_sync(gmask, nbSym, slot * 4);
  if (e) return false;
  huf_fill_root(sm.root[slot], R, wk, slotMem, tl, nbSym, sub, 4);
  if (tl > R) huf_fill_table(fullMem, (u8*)(fullMem + (1u << HUF_TABLE_LOG)), wk, slotMem, tl, nbSym, sub, 4, R);
  __syncwarp(gmask);
  T.full = fullMem; T.side = (const u8*)(fullMem + (1u << HUF_TABLE_LOG)); T.log = tl;
  *hdrOut = hdr;
  return true;
}
// the dictionary's table (litEntropy = 1 after ZSTD_decompress_insertDictionary, :2468)
template <int R>
__device__ __forceinline__ void huf_dict_tables(HufSmem<R>& sm, u32 slot, u32 sub, unsigned gmask, const DictState* ds, HufTabs& T) {
  huf_root_from_full(sm.root[slot], R, ds->huf, ds->hufLog, sub, 4);
  __syncwarp(gmask);
  T.full = ds->huf; T.side = ds->hufSide; T.log = ds->hufLog;
}

// one frame by its 4-lane group
template <int R>
__device__ __forceinline__ void huf_frame(const DecodeArgs& a, HufSmem<R>& sm, u32 f, u32 lane, u16* fullMem) {
  const u32 sub = lane & 3, slot = lane >> 2;
  const unsigned gmask = 0xFu << (slot * 4);
  const FrameInfo fi = a.info[f];
  if (fi.flags & (FI_DONE | FI_PAR)) return;   // whole 4-lane group leaves together; group syncs below use gmask
  if (((fi.flags & FI_SMALLHUF) != 0) != (R == (int)HUF_ROOT_SMALL)) return;       // the other instantiation's frame
  const u8* src = a.src_base + a.src_off[f]; const u32 size = a.src_size[f];
  u8* lit = lit_region(a, f, fi); const u64 litCap = lit_capacity(frame_cap(a, f, fi));
  u32 pos = fi.body_off, blk = 0; u64 litRun = 0;
  HufTabs T{sm.root[slot], R, nullptr, nullptr, 0}; bool haveTable = false;
  __syncwarp(gmask);                                                               // the group's previous frame is done with root / rings
  if (a.dict && a.dict->hasEntropy) { huf_dict_tables(sm, slot, sub, gmask, a.dict, T); haveTable = true; }
  u32 errBlock = 0xFFFFFFFFu, errCode = 0;
  while (true) {
    BlockHdr bh;
    if (read_block_hdr(src + pos, size - pos, bh)) break;
    pos += 3;
    if (bh.type == 2) {
      const u8* bp = src + pos; u32 bsz = bh.csize;
      if (bsz >= BLOCKSIZE_MAX) break;
      LitHdr lh; bool needs;
      if (read_lit_hdr(bp, bsz, lh, &needs)) break;
      if (lh.type >= 2) {
        if (lh.type == 3 && !haveTable) break;                                     // dictionary_corrupted, reported by k_exec
        bool ok = true;
        const u8* body = bp + lh.lhSize; u32 bodySize = lh.litCSize;
        const bool dry = litRun + lh.litSize + 3 > litCap;                         // cannot be stored: validate only (HUF_DRY)
        if (lh.type == 2) {
          if (!lh.single && (lh.litSize == 0 || bodySize == 0)) ok = false;       // HufDecompress.cs:1211-1212
          u32 hdr = 0;
          if (ok) ok = huf_build_tables(sm, slot, sub, gmask, body, bodySize, fullMem, T, &hdr);
          if (ok) { body += hdr; bodySize -= hdr; haveTable = true; }
        }
        if (ok) {
          bool good = true;
          if (lh.single) {
            if (sub == 0) good = dry ? huf_check_stream(body, bodySize, lh.litSize, T)
                                     : huf_decode_stream(body, bodySize, lit + litRun, lh.litSize, T, &sm.ring[lane][0]);   // HufDecompress.cs:247-264
          } else {
            HufStream st;
            good = huf_split4(body, bodySize, lh.litSize, sub, st);
            if (good) good = dry ? huf_check_stream(st.src, st.len, st.count, T)
                                 : huf_decode_stream(st.src, st.len, lit + litRun + st.outOfs, st.count, T, &sm.ring[lane][0]);
          }
          unsigned okmask = __ballot_sync(gmask, good);
          if ((okmask & gmask) != gmask) ok = false;
          __syncwarp(gmask);                                                       // the rings are free again (a later block's weights use them)
        }
        if (!ok || dry) { errBlock = blk; errCode = ok ? HUF_DRY : ZE_corruption_detected; break; }
        litRun += lh.litSize;
      }
    }
    pos += bh.csize; blk++;
    if (bh.last) break;
  }
  if (sub == 0 && errBlock != 0xFFFFFFFFu) { a.info[f].huf_err_block = errBlock; a.info[f].huf_err_code = errCode; }
}

// persistent: grid = the CTAs one wave of the device holds (or fewer for small batches)
template <int R>
__global__ void __launch_bounds__(32) k_huf(DecodeArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  HufSmem<R>& sm = *reinterpret_cast<HufSmem<R>*>(smem_raw);
  const u32 lane = threadIdx.x, slot = lane >> 2;
  const u32 nSmall = a.cnt[2];                                                     // frames k_parse marked FI_SMALLHUF
  if (R == (int)HUF_ROOT_SMALL ? nSmall == 0 : nSmall == a.n) return;              // nothing for this instantiation in the launch
  u16* const fullMem = a.huf_full + (size_t)(blockIdx.x * 8 + slot) * HUF_FULL_STRIDE;
  for (u32 g = blockIdx.x; g * 8 < a.n; g += gridDim.x) {
    const u32 f = g * 8 + slot;
    if (f < a.n) huf_frame(a, sm, f, lane, fullMem);
  }
}

// =================================================================================================
// k_seq : one warp per CTA, one frame per lane, tables bank-interleaved across lanes
// =================================================================================================
// The chain half (seq_decode_frame) and the finishing half (SeqEmitter) of sequence decoding run in the same thread.
// (Measured alternative, round 2: the two halves on two warps of a CTA — two schedulers — joined by a per-lane
// shared-memory queue.  The chain warp's loop went from 136 to 103 instructions but only from ~400 to ~373 cycles per
// sequence: it is bound by the dependent chain state -> cell -> extra-bit count -> shift -> state plus the one-warp ALU
// issue rate, and the queue's back-pressure test adds a divergent branch; 2.06 ms against 1.72 ms for this kernel.)
// CL / CO / CM: the largest table logs the instantiation has room for.  Three instantiations share the frames (k_parse
// classifies them by the first block's sequence count, which bounds the table logs every known encoder chooses):
// 6 / 6 / 7 (32 KB, 6 CTAs per SM), 8 / 8 / 8 (64 KB, 3 CTAs per SM) and the format's maximum 9 / 8 / 9 (98 KB, 2 CTAs per SM).
// A frame that turns out to need a larger table than its class provides is handed to the full-size instantiation, which
// runs last (SeqEmitter::defer).
template <int CL, int CO, int CM> struct SeqSmemT {
  u16 ll[1 << CL][32];   // lane-interleaved: cell[state][lane]
  u16 ml[1 << CM][32];
  u16 of[1 << CO][32];
  u16 defLL[64], defOF[32], defML[64];
  u32 llInfo[36], mlInfo[53];
  s16 norm[53][32];      // per-lane scratch of the table builder, lane-interleaved like the tables
  u16 next[53][32];
  __align__(16) u32 ring[32][ZB_RING_WORDS + 4];   // per-lane bitstream read-ahead (BitRing), skewed by 4 banks per lane
};
typedef SeqSmemT<9, 8, 9> SeqSmem;

template <class SM>
__device__ __forceinline__ void seq_smem_init(SM& sm, u32 lane) {
  // predefined tables + info LUTs, built once per CTA
  if (lane < 3) {
    s16* norm = &sm.norm[0][lane]; u16* next = &sm.next[0][lane];
    Strided<s16> nv{norm, 32}; Strided<u16> sn{next, 32};
    if (lane == 0) { for (int i = 0; i < 36; i++) nv[i] = kLLnorm[i]; build_seq_table(sm.defLL, 1, nv, 35, 6, sn); }
    if (lane == 1) { for (int i = 0; i < 29; i++) nv[i] = kOFnorm[i]; build_seq_table(sm.defOF, 1, nv, 28, 5, sn); }
    if (lane == 2) { for (int i = 0; i < 53; i++) nv[i] = kMLnorm[i]; build_seq_table(sm.defML, 1, nv, 52, 6, sn); }
  }
  for (u32 i = lane; i < 36; i += 32) sm.llInfo[i] = ll_info(i);
  for (u32 i = lane; i < 53; i += 32) sm.mlInfo[i] = ml_info(i);
  __syncwarp();
}

// CLS: 0 = full-size tables (also every frame the smaller instantiations handed over), 1 = FI_SEQ_A, 2 = FI_SEQ_B
template <int CLS, int CL, int CO, int CM>
__global__ void __launch_bounds__(32) k_seq_t(DecodeArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  typedef SeqSmemT<CL, CO, CM> SM;
  SM& sm = *reinterpret_cast<SM*>(smem_raw);
  const u32 lane = threadIdx.x;
  // this class's frames: a dense list written by k_parse; the full-size class also gets what the smaller ones handed over
  const u32 k = CLS == 0 ? 2 : CLS - 1;
  const u32 count = a.cnt[3 + k];
  if (blockIdx.x * 32 >= count) return;
  seq_smem_init(sm, lane);
  const u32 e = blockIdx.x * 32 + lane;
  if (e >= count) return;
  const u32 f = a.par_list[(size_t)(1 + k) * a.list_stride + a.item_base + e];
  const FrameInfo fi = a.info[f];
  SeqTableSet T;
  T.cap[KIND_LL] = CL; T.cap[KIND_OF] = CO; T.cap[KIND_ML] = CM;
  T.space[KIND_LL] = &sm.ll[0][lane]; T.space[KIND_ML] = &sm.ml[0][lane]; T.space[KIND_OF] = &sm.of[0][lane]; T.stride = 32;
  T.defs[KIND_LL] = sm.defLL; T.defs[KIND_OF] = sm.defOF; T.defs[KIND_ML] = sm.defML;
  SeqEmitter em;
  em.init(seq_region(a, f, fi), seq_capacity(frame_cap(a, f, fi)), sm.llInfo, sm.mlInfo);
  if (a.dict) em.set_reps(a.dict->rep);
  seq_decode_frame(a.src_base + a.src_off[f], a.src_size[f], fi.body_off, fi.window, T, em, sm.llInfo, sm.mlInfo,
                   Strided<s16>{&sm.norm[0][lane], 32}, Strided<u16>{&sm.next[0][lane], 32}, &sm.ring[lane][0], a.dict);
  if (CLS != 0 && em.deferred) {                                                   // the full-size instantiation (launched after this one) redoes the frame
    a.info[f].flags = fi.flags & ~(u32)(FI_SEQ_A | FI_SEQ_B);
    a.par_list[(size_t)3 * a.list_stride + a.item_base + atomicAdd(a.cnt + 5, 1u)] = f;
    return;
  }
  if (em.res.err_block != 0xFFFFFFFFu) {
    a.info[f].seq_err_block = em.res.err_block; a.info[f].seq_err_code = em.res.err_code; a.info[f].seq_err_index = em.res.err_index;
  }
}

// =================================================================================================
// warp-cooperative byte movers
// =================================================================================================
// dst and src must not overlap.  All 32 lanes call with identical arguments.
__device__ __forceinline__ void warp_copy(u8* dst, const u8* src, u32 n, u32 lane) {
  if (n < 128) { for (u32 i = lane; i < n; i += 32) dst[i] = src[i]; return; }
  u32 head = (u32)(-(intptr_t)dst) & 15;
  if (lane < head) dst[lane] = src[lane];
  dst += head; src += head; n -= head;
  u32 body = n & ~15u;
  if ((((uintptr_t)src) & 15) == 0) {
    const uint4* s = (const uint4*)src; uint4* d = (uint4*)dst;
    for (u32 i = lane; i < body / 16; i += 32) d[i] = s[i];
  } else {
    // dst is 16-byte aligned, src is not: rebuild each 16-byte vector from five aligned 4-byte words of src
    const u32 sh = ((u32)(uintptr_t)src & 3) * 8;
    const u32* s = (const u32*)((uintptr_t)src & ~(uintptr_t)3); uint4* d = (uint4*)dst;
    for (u32 i = lane; i < body / 16; i += 32) {
      const u32* p = s + 4 * i;
      u32 w0 = p[0], w1 = p[1], w2 = p[2], w3 = p[3], w4 = sh ? p[4] : 0;
      d[i] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
    }
  }
  for (u32 i = body + lane; i < n; i += 32) dst[i] = src[i];
}
__device__ __forceinline__ void warp_fill(u8* dst, u8 v, u32 n, u32 lane) {
  if (n < 128) { for (u32 i = lane; i < n; i += 32) dst[i] = v; return; }
  u32 head = (u32)(-(intptr_t)dst) & 15;
  if (lane < head) dst[lane] = v;
  dst += head; n -= head;
  u32 body = n & ~15u, w = v * 0x01010101u;
  uint4* d = (uint4*)dst; uint4 vv = make_uint4(w, w, w, w);
  for (u32 i = lane; i < body / 16; i += 32) d[i] = vv;
  for (u32 i = body + lane; i < n; i += 32) dst[i] = v;
}

__device__ __forceinline__ u32 warp_incl_scan(u32 v, u32 lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { u32 t = __shfl_up_sync(0xFFFFFFFFu, v, d); if (lane >= (u32)d) v += t; }
  return v;
}

// =================================================================================================
// k_exec : one warp per frame
// =================================================================================================
// Sequence execution is the reference's ExecSequence loop (:1265-1352, :1582-1605) re-expressed for a warp:
// 32 sequence records are taken at a time, one per lane.  Output positions come from a warp prefix sum, all
// literal runs of the group are copied first (they depend on nothing), then matches are resolved in rounds: a
// match is ready once every earlier match of the group whose output overlaps its source has been written
// (sources before the group are always ready).  Ready matches of a round are copied together, one output byte
// per lane, by mapping a flattened byte index back to its sequence with a shuffle binary search.  Matches that
// overlap their own output (offset < length) or are long are handled one at a time by the whole warp.
#define FULLMASK 0xFFFFFFFFu

// number of lanes whose inclusive prefix `incl` (non-decreasing over lanes) is <= x; x may differ per lane.
// Saturates at 31: callers only ask for x < incl[31].
__device__ __forceinline__ u32 warp_upper_bound(u32 incl, u32 x) {
  u32 j = 0;
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) { u32 v = __shfl_sync(FULLMASK, incl, j + s - 1); if (v <= x) j += s; }
  return j;   // j + s - 1 <= 30 inside the loop and j <= 31 here: no lane index ever wraps
}

// Flattened copy of many short runs in units of one 4-byte-aligned destination word: run of lane j writes len_j
// bytes at g + dpos_j, i.e. touches units_j = ((g + dpos_j) % 4 + len_j + 3) / 4 aligned words (the first and the
// last possibly in part); uincl/uexcl are the inclusive/exclusive warp prefix sums of units_j.  One unit per
// lane and row, U rows in flight per pass so that the U shuffle binary searches and the U loads overlap instead
// of serialising on their latencies.  Source of run j: src + spos_j.  The source word is assembled from the (at
// most two) aligned words that hold a byte the unit needs — nothing outside [source, source + len_j) rounded to
// words is touched.  (Used for literal runs; the same scheme for matches measured slower than flat_copy_m4.)
template <int U>
__device__ __forceinline__ void flat_copy_w(u8* g, const u8* src, u32 totalUnits, u32 uincl, u32 uexcl, u32 dpos, u32 spos, u32 len, u32 lane) {
  for (u32 t0 = 0; t0 < totalUnits; t0 += 32 * U) {
    u32 t[U], j[U], dj[U], ej[U], sj[U], nj[U], v[U], lo[U], hi[U];
#pragma unroll
    for (int k = 0; k < U; k++) { t[k] = t0 + 32 * k + lane; j[k] = 0; }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
#pragma unroll
      for (int k = 0; k < U; k++) { const u32 x = __shfl_sync(FULLMASK, uincl, j[k] + s - 1); if (x <= t[k]) j[k] += s; }
    }
#pragma unroll
    for (int k = 0; k < U; k++) {
      dj[k] = __shfl_sync(FULLMASK, dpos, j[k]); ej[k] = __shfl_sync(FULLMASK, uexcl, j[k]);
      sj[k] = __shfl_sync(FULLMASK, spos, j[k]); nj[k] = __shfl_sync(FULLMASK, len, j[k]);
    }
#pragma unroll
    for (int k = 0; k < U; k++) {
      v[k] = 0; lo[k] = 0; hi[k] = 0;
      if (t[k] < totalUnits) {
        u8* const d0 = g + dj[k];                                         // first byte of the run
        const u32 word = ((u32)(uintptr_t)d0 & 3) + 0;                    // its position within its aligned word
        const i32 rel = (i32)(4 * (t[k] - ej[k])) - (i32)word;           // run-relative position of this unit's word (-3..)
        lo[k] = rel < 0 ? (u32)-rel : 0;                                  // bytes [lo, hi) of the word belong to the run
        const u32 left = nj[k] - (u32)(rel + (i32)lo[k]);
        hi[k] = lo[k] + left < 4 ? lo[k] + left : 4;
        const u8* sp = src + sj[k] + rel;                                 // source of the word's byte 0
        const u32* w = (const u32*)((uintptr_t)sp & ~(uintptr_t)3); const u32 sb = (u32)(uintptr_t)sp & 3;
        const u32 a0 = (sb + lo[k] < 4) ? w[0] : 0, a1 = (sb + hi[k] > 4) ? w[1] : 0;
        v[k] = __funnelshift_r(a0, a1, sb * 8);
      }
    }
#pragma unroll
    for (int k = 0; k < U; k++) if (t[k] < totalUnits) {
      u8* d = (u8*)(((uintptr_t)(g + dj[k]) & ~(uintptr_t)3) + 4 * (size_t)(t[k] - ej[k]));
      if (hi[k] - lo[k] == 4) *(u32*)d = v[k];
      else {
        if (lo[k] == 0) d[0] = (u8)v[k];
        if (lo[k] <= 1 && hi[k] > 1) d[1] = (u8)(v[k] >> 8);
        if (lo[k] <= 2 && hi[k] > 2) d[2] = (u8)(v[k] >> 16);
        if (hi[k] == 4) d[3] = (u8)(v[k] >> 24);
      }
    }
  }
}
// RLE literals: the same units, filled with one byte value
template <int U>
__device__ __forceinline__ void flat_fill_w(u8* g, u32 fillWord, u32 totalUnits, u32 uincl, u32 uexcl, u32 dpos, u32 len, u32 lane) {
  for (u32 t0 = 0; t0 < totalUnits; t0 += 32 * U) {
#pragma unroll
    for (int k = 0; k < U; k++) {
      const u32 t = t0 + 32 * k + lane; u32 j = 0;
#pragma unroll
      for (int s = 16; s >= 1; s >>= 1) { const u32 x = __shfl_sync(FULLMASK, uincl, j + s - 1); if (x <= t) j += s; }
      const u32 dj = __shfl_sync(FULLMASK, dpos, j), ej = __shfl_sync(FULLMASK, uexcl, j), nj = __shfl_sync(FULLMASK, len, j);
      if (t < totalUnits) {
        u8* const d0 = g + dj;
        const i32 rel = (i32)(4 * (t - ej)) - (i32)((u32)(uintptr_t)d0 & 3);
        const u32 lo = rel < 0 ? (u32)-rel : 0, left = nj - (u32)(rel + (i32)lo), hi = lo + left < 4 ? lo + left : 4;
        u8* d = (u8*)(((uintptr_t)d0 & ~(uintptr_t)3) + 4 * (size_t)(t - ej));
        if (hi - lo == 4) *(u32*)d = fillWord;
        else for (u32 b = lo; b < hi; b++) d[b] = (u8)fillWord;
      }
    }
  }
}
// units of a run of len bytes starting at p (0 for an empty run)
__device__ __forceinline__ u32 word_units(const u8* p, u32 len) { return len ? (((u32)(uintptr_t)p & 3) + len + 3) >> 2 : 0; }

// Flattened copy of many short non-overlapping matches in units of 4 bytes: run of lane j has len_j bytes
// (off_j >= len_j), i.e. (len_j + 3) / 4 units; unit u moves bytes [4u, min(4u + 4, len_j)) from g + mrel_j - off_j.
// The source word is assembled from two aligned loads (bytes past the run's end are read and dropped).
template <int U>
__device__ __forceinline__ void flat_copy_m4(u8* g, u32 totalUnits, u32 uincl, u32 uexcl, u32 mrel, u32 off, u32 len, u32 lane) {
  for (u32 t0 = 0; t0 < totalUnits; t0 += 32 * U) {
    u32 t[U], j[U], dj[U], ej[U], oj[U], nj[U], v[U];
#pragma unroll
    for (int k = 0; k < U; k++) { t[k] = t0 + 32 * k + lane; j[k] = 0; }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
#pragma unroll
      for (int k = 0; k < U; k++) { const u32 x = __shfl_sync(FULLMASK, uincl, j[k] + s - 1); if (x <= t[k]) j[k] += s; }
    }
#pragma unroll
    for (int k = 0; k < U; k++) {
      dj[k] = __shfl_sync(FULLMASK, mrel, j[k]); ej[k] = __shfl_sync(FULLMASK, uexcl, j[k]);
      oj[k] = __shfl_sync(FULLMASK, off, j[k]); nj[k] = __shfl_sync(FULLMASK, len, j[k]);
    }
#pragma unroll
    for (int k = 0; k < U; k++) {
      v[k] = 0;
      if (t[k] < totalUnits) {
        const u8* sp = g + dj[k] + 4 * (t[k] - ej[k]) - (size_t)oj[k];
        const u32* w = (const u32*)((uintptr_t)sp & ~(uintptr_t)3); const u32 sh = ((u32)(uintptr_t)sp & 3) * 8;
        const u32 a0 = w[0], a1 = sh ? w[1] : 0;
        v[k] = __funnelshift_r(a0, a1, sh);
      }
    }
#pragma unroll
    for (int k = 0; k < U; k++) if (t[k] < totalUnits) {
      const u32 b0 = 4 * (t[k] - ej[k]); const u32 cnt = nj[k] - b0;   // >= 1
      u8* d = g + dj[k] + b0;
      if (cnt >= 4 && (((uintptr_t)d) & 3) == 0) *(u32*)d = v[k];
      else { d[0] = (u8)v[k]; if (cnt > 1) d[1] = (u8)(v[k] >> 8); if (cnt > 2) d[2] = (u8)(v[k] >> 16); if (cnt > 3) d[3] = (u8)(v[k] >> 24); }
    }
  }
}

// one match copied by the whole warp; handles every offset/length relation (byte-serial semantics of :1319-1350)
__device__ __forceinline__ void warp_match(u8* d, u32 off, u32 len, u32 lane) {
  const u8* s = d - off;
  if (off >= len) { warp_copy(d, s, len, lane); return; }
  if (off >= 32) {
    for (u32 i0 = 0; i0 < len; i0 += 32) { u32 i = i0 + lane; if (i < len) d[i] = s[i]; __syncwarp(); }
    return;
  }
  u32 r = lane % off; const u32 stepm = 32 % off;          // period-`off` pattern: byte i repeats byte i mod off
  for (u32 i = lane; i < len; i += 32) { d[i] = s[r]; r += stepm; if (r >= off) r -= off; }
}

// 16 CTAs of 4 warps per SM (32 registers, spills to local memory included): measured faster than fewer, fatter warps —
// the kernel lives on occupancy (6 / 8 / 10 / 12 / 16 CTAs: 3.93 / 3.44 / 3.03 / 2.95 / 2.83 ms on the bench workload).
// DICT: the context has a dictionary (its content is the window's prefix); the common kernel carries none of that code
template <bool DICT>
__global__ void __launch_bounds__(EXEC_THREADS, 16) k_exec(DecodeArgs a) {
  const u32 lane = threadIdx.x & 31;
  const u32 f = (blockIdx.x * EXEC_THREADS + threadIdx.x) >> 5;
  if (f >= a.n) return;
  FrameInfo fi = a.info[f];
  if (fi.flags & (FI_DONE | FI_PAR)) return;
  const u8* src = a.src_base + a.src_off[f]; const u32 size = a.src_size[f];
  u8* dst = a.dst_base + frame_dst_off(a, f, fi); const u32 cap = frame_cap(a, f, fi);
  const u8* litScratch = lit_region(a, f, fi);
  const SeqRec* recs = seq_region(a, f, fi); const u32 recCap = (u32)seq_capacity(cap);
  u32 pos = fi.body_off, blk = 0, op = 0, litRun = 0, recRun = 0;   // op <= cap < 2^32 throughout: checks are written against cap - op
  bool litEntropy = false, dry = false; u32 err = 0;
  // the dictionary's content is the window's prefix (RefDictContent :2366-2373): dictEnd[-k] is what offset (produced + k) reaches
  const u32 dictContent = DICT ? a.dict->contentSize : 0;
  const u8* const dictEnd = DICT ? a.dict_bytes + a.dict->contentOff + dictContent : nullptr;
  if (DICT && a.dict->hasEntropy) litEntropy = true;                               // :2468
  while (true) {
    BlockHdr bh;
    err = read_block_hdr(src + pos, size - pos, bh);
    if (err) break;
    pos += 3;
    if (bh.type == 0) {                                                            // raw, :662-667
      if (bh.csize > cap - op) { err = ZE_dstSize_tooSmall; break; }
      warp_copy(dst + op, src + pos, bh.csize, lane); op += bh.csize;
    } else if (bh.type == 1) {                                                     // RLE, :1945-1950
      if (bh.orig > cap - op) { err = ZE_dstSize_tooSmall; break; }
      warp_fill(dst + op, src[pos], bh.orig, lane); op += bh.orig;
    } else {
      const u8* bp = src + pos; const u32 bsz = bh.csize;
      if (bsz >= BLOCKSIZE_MAX) { err = ZE_srcSize_wrong; break; }                 // :1880
      LitHdr lh; bool needs;
      u32 e = read_lit_hdr(bp, bsz, lh, &needs);
      if (needs && !litEntropy) { err = ZE_dictionary_corrupted; break; }          // :696-697
      if (e) { err = e; break; }
      const u8* lit; u32 rleByte = 0; bool isRle = false;
      if (lh.type >= 2) {
        if (fi.huf_err_block == blk) {
          if (fi.huf_err_code != HUF_DRY) { err = fi.huf_err_code; break; }        // :742 (all Huffman failures -> corruption_detected)
          dry = true;                                                              // literals were not stored: checks only, the block must fail
        }
        litEntropy = true; lit = litScratch + litRun; litRun += lh.litSize;
      } else if (lh.type == 0) lit = bp + lh.lhSize;
      else { lit = nullptr; isRle = true; rleByte = bp[lh.lhSize]; }
      const u32 litSize = lh.litSize;
      const u8* sp = bp + lh.consumed; const u32 ssz = bsz - lh.consumed;
      u32 nbSeq, modes, hdr;
      e = read_seq_count(sp, ssz, &nbSeq, &modes, &hdr);
      if (e) { err = e; break; }
      if (fi.seq_err_block == blk && fi.seq_err_index == 0xFFFFFFFFu) { err = fi.seq_err_code; break; }
      u32 litPos = 0;
      if (nbSeq) {
        // the block's header record: how many records follow and what they produce (zb_decode.cuh)
        u32 nRecs = 0, outBytes = 0, litBytes = 0;
        if (recRun < recCap) { const uint4 h = __ldg(reinterpret_cast<const uint4*>(recs + recRun)); nRecs = h.x; outBytes = h.y; litBytes = h.z; }
        const uint4* rv = reinterpret_cast<const uint4*>(recs + recRun + 1);
        const u32 blockBase = op;
        for (u32 g0 = 0; g0 < nRecs; g0 += 32) {
          const bool valid = g0 + lane < nRecs;
          const uint4 rec = valid ? __ldg(rv + g0 + lane) : make_uint4(0, 0, 0, 0);
          if (lane < 2 && g0 + 32 < nRecs) prefetch_line(rv + g0 + 32 + 16 * lane);   // next group's 512 bytes
          const u32 ll = valid ? (rec.w & 0x1FFFF) : 0, ml = valid ? ((rec.w >> 17) | (((rec.y >> 18) & 7) << 15)) : 0, off = rec.z, lpos = rec.y & 0x3FFFF;
          // checks in the reference's order (:1278, :1279, :1290-1294)
          const u64 start64 = (u64)blockBase + rec.x;
          const bool e1 = valid && start64 + ll + ml > cap;
          const bool e2 = valid && lpos + ll > litSize;
          const bool e3 = valid && (u64)off > start64 + ll + dictContent;           // :1290-1294 (the prefix includes the dictionary)
          const unsigned bad = __ballot_sync(FULLMASK, e1 | e2 | e3);
          if (bad) {
            const u32 first = (u32)__ffs(bad) - 1;
            const u32 code = e1 ? ZE_dstSize_tooSmall : ZE_corruption_detected;
            err = __shfl_sync(FULLMASK, code, first);
            break;
          }
          // group-relative positions straight from the records (no prefix sums): the group writes at g = dst + op
          const u32 base = __shfl_sync(FULLMASK, rec.x, 0), lbase = __shfl_sync(FULLMASK, lpos, 0);
          op = blockBase + base; litPos = lbase;
          const u32 excl = valid ? rec.x - base : 0, mrel = excl + ll, incl = valid ? mrel + ml : 0xFFFFFFFFu;   // lanes past the end never bound a search
          const u32 lsrc = lpos - lbase;                    // literal source position of this lane, relative to litPos
          u8* const g = dst + op;
          // ---- literals: short runs flattened over the lanes, long runs by the whole warp ----
          if (!dry) {
            const bool bigL = ll >= 128;
            unsigned bigMask = __ballot_sync(FULLMASK, bigL);
            const u32 ls = bigL ? 0 : ll;
            const u32 lu = word_units(g + excl, ls);
            const u32 sincl = warp_incl_scan(lu, lane), sexcl = sincl - lu;
            const u32 Ls = __shfl_sync(FULLMASK, sincl, 31);
            if (isRle) { if (Ls) flat_fill_w<1>(g, rleByte * 0x01010101u, Ls, sincl, sexcl, excl, ls, lane); }
            else if (Ls > 32) flat_copy_w<2>(g, lit + litPos, Ls, sincl, sexcl, excl, lsrc, ls, lane);
            else if (Ls) flat_copy_w<1>(g, lit + litPos, Ls, sincl, sexcl, excl, lsrc, ls, lane);
            while (bigMask) {
              const u32 j = (u32)__ffs(bigMask) - 1; bigMask &= bigMask - 1;
              const u32 dj = __shfl_sync(FULLMASK, excl, j), nj = __shfl_sync(FULLMASK, ll, j), lj = __shfl_sync(FULLMASK, lsrc, j);
              if (isRle) warp_fill(g + dj, (u8)rleByte, nj, lane); else warp_copy(g + dj, lit + litPos + lj, nj, lane);
            }
          }
          __syncwarp();
          // ---- matches, in dependency rounds ----
          const bool hasM = ml > 0 && off != 0;               // offset 0 (corrupted input only) copies bytes onto themselves
          const unsigned matchMask = __ballot_sync(FULLMASK, hasM);
          if (matchMask && !dry) {
            unsigned depMask = 0;
            {
              const i64 slo = (i64)mrel - (i64)off;                         // source range, group-relative
              i64 shi = slo + (i64)ml; if (shi > (i64)mrel) shi = (i64)mrel;   // own output is handled by warp_match
              const bool dep = hasM && shi > 0;
              const u32 needLo = slo > 0 ? (u32)slo : 0, needHi = dep ? (u32)shi : 1;
              const u32 aIdx = warp_upper_bound(incl, dep ? needLo : 0), bIdx = warp_upper_bound(incl, needHi - 1);
              if (dep) {
                const unsigned upTo = bIdx >= 31 ? 0xFFFFFFFFu : ((1u << (bIdx + 1)) - 1);
                depMask = upTo & ~((1u << aIdx) - 1) & ((1u << lane) - 1) & matchMask;
              }
            }
            unsigned doneMask = ~matchMask;
            while (doneMask != 0xFFFFFFFFu) {
              const bool ready = hasM && !((doneMask >> lane) & 1) && ((depMask & ~doneMask) == 0);
              const unsigned R = __ballot_sync(FULLMASK, ready);
              const bool inDict = DICT && off > blockBase + base + mrel;          // the source begins in the dictionary (:1290-1315)
              const bool plain = ready && off >= ml && ml < 128 && !inDict;
              const u32 len = plain ? ml : 0, units = (len + 3) >> 2;
              const u32 pincl = warp_incl_scan(units, lane), pexcl = pincl - units;
              const u32 Tt = __shfl_sync(FULLMASK, pincl, 31);
              if (Tt > 32) flat_copy_m4<2>(g, Tt, pincl, pexcl, mrel, off, len, lane);
              else if (Tt) flat_copy_m4<1>(g, Tt, pincl, pexcl, mrel, off, len, lane);
              unsigned big = __ballot_sync(FULLMASK, ready && !plain);
              while (big) {
                const u32 j = (u32)__ffs(big) - 1; big &= big - 1;
                const u32 mj = __shfl_sync(FULLMASK, mrel, j), oj = __shfl_sync(FULLMASK, off, j), nj = __shfl_sync(FULLMASK, ml, j);
                const u32 pj = blockBase + base + mj;                              // the match's output position within the frame
                if (DICT && oj > pj) {
                  // `back` bytes come from the end of the dictionary content, the rest continues at the frame's first byte
                  const u32 back = oj - pj, l1 = back < nj ? back : nj;
                  warp_copy(g + mj, dictEnd - back, l1, lane);
                  __syncwarp();
                  if (nj > l1) warp_match(g + mj + l1, pj + l1, nj - l1, lane);
                } else warp_match(g + mj, oj, nj, lane);
              }
              __syncwarp();
              doneMask |= R;
            }
          }
        }
        if (err) break;
        recRun += 1 + nRecs;
        if (fi.seq_err_block == blk) { err = fi.seq_err_code; break; }             // :1594 after the decodable prefix
        op = blockBase + outBytes; litPos = litBytes;
      }
      // last literals (:1599-1605)
      const u32 lastLL = litSize - litPos;
      if (lastLL > cap - op || dry) { err = ZE_dstSize_tooSmall; break; }
      if (isRle) warp_fill(dst + op, (u8)rleByte, lastLL, lane); else warp_copy(dst + op, lit + litPos, lastLL, lane);
      op += lastLL;
      __syncwarp();
    }
    pos += bh.csize; blk++;
    if (bh.last) break;
  }
  // ---- frame epilogue (:2069-2085) and the multi-frame loop tail (:2111-2157) ----
  bool needXxh = false; u32 trailer = 0;
  if (!err) {
    if ((fi.flags & FI_FCS_KNOWN) && op != fi.fcs) err = ZE_corruption_detected;
    else if (fi.flags & FI_CHECKSUM) {
      if (size - pos < 4) err = ZE_checksum_wrong; else { trailer = pos; pos += 4; needXxh = true; }
    }
  }
  u32 tailErr = 0, nextOff = 0;
  if (!err) {
    while (true) {
      u32 rem = size - pos;
      if (rem < 5) { if (rem) tailErr = ZE_srcSize_wrong; break; }
      u32 magic = ld32(src + pos);
      if (magic == MAGIC) { nextOff = pos; break; }                                // another data frame: next pass (:2111-2153)
      if ((magic & 0xFFFFFFF0u) != MAGIC_SKIP) { tailErr = ZE_prefix_unknown; break; }
      if (rem < 8) { tailErr = ZE_srcSize_wrong; break; }
      u32 skip = ld32(src + pos + 4) + 8u;
      if (rem < skip) { tailErr = ZE_srcSize_wrong; break; }
      pos += skip;
    }
  }
  if (lane == 0) {
    u32 res = err ? zerr(err) : (tailErr ? zerr(tailErr) : fi.out_base + (u32)op);
    a.result[f] = res;                                                             // provisional while next_off != 0
    a.info[f].trailer_off = trailer; a.info[f].decoded = (u32)op; a.info[f].next_off = nextOff;
    a.info[f].flags = fi.flags | (needXxh ? FI_NEED_XXH : 0);
    if (nextOff && a.more) atomicAdd(a.more, 1u);
  }
}

// =================================================================================================
// Block-parallel path for multi-block frames (zb_blocks.cuh): every compressed block of an FI_PAR frame is a unit
// =================================================================================================
// k_huf_blk : k_huf's mapping (4 lanes per unit, 8 units per warp), persistent over the launch's units
__global__ void __launch_bounds__(32) k_huf_blk(DecodeArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  HufSmem<HUF_TABLE_LOG>& sm = *reinterpret_cast<HufSmem<HUF_TABLE_LOG>*>(smem_raw);
  const u32 lane = threadIdx.x, sub = lane & 3, slot = lane >> 2;
  const unsigned gmask = 0xFu << (slot * 4);
  const u32 nunits = a.cnt[0];
  BlockUnit* const sliceUnits = a.units + unit_slice_base(a);
  u16* const fullMem = a.huf_full + (size_t)(blockIdx.x * 8 + slot) * HUF_FULL_STRIDE;
  for (u32 w0 = blockIdx.x * 8; w0 < nunits; w0 += gridDim.x * 8) {
    const u32 w = w0 + slot;
    if (w >= nunits) continue;                                                     // the whole 4-lane group together
    const BlockUnit u = sliceUnits[w];
    const u32 f = u.frame;
    const FrameInfo fi = a.info[f];
    const u8* src = a.src_base + a.src_off[f];
    const u8* bp = src + u.body;
    LitHdr lh; bool needs;
    read_lit_hdr(bp, u.csize, lh, &needs);                                         // sound: par_walk has parsed it
    if (lh.type < 2) continue;
    u8* lit = lit_region(a, f, fi) + u.lit_off;
    bool ok = true;
    HufTabs T{sm.root[slot], HUF_TABLE_LOG, nullptr, nullptr, 0};
    const u8* body = bp + lh.lhSize; u32 bodySize = lh.litCSize;
    __syncwarp(gmask);                                                             // the group's previous unit is done with root / rings
    if (lh.type == 3 && u.huf_def == DEF_DICT) huf_dict_tables(sm, slot, sub, gmask, a.dict, T);
    else {
      // the weights: this block's own (type 2) or those of the block that defined the table in force (treeless)
      const u8* tb = body; u32 tbSize = bodySize;
      if (lh.type == 3) {
        const BlockUnit d = sliceUnits[fi.unit_base + u.huf_def];
        LitHdr lhD; bool n2;
        read_lit_hdr(src + d.body, d.csize, lhD, &n2);
        tb = src + d.body + lhD.lhSize; tbSize = lhD.litCSize;
      } else if (!lh.single && (lh.litSize == 0 || bodySize == 0)) ok = false;     // HufDecompress.cs:1211-1212
      u32 hdr = 0;
      if (ok) ok = huf_build_tables(sm, slot, sub, gmask, tb, tbSize, fullMem, T, &hdr);
      if (ok && lh.type == 2) { body += hdr; bodySize -= hdr; }
    }
    if (ok) {
      bool good = true;
      if (lh.single) {
        if (sub == 0) good = huf_decode_stream(body, bodySize, lit, lh.litSize, T, &sm.ring[lane][0]);
      } else {
        HufStream st;
        good = huf_split4(body, bodySize, lh.litSize, sub, st);
        if (good) good = huf_decode_stream(st.src, st.len, lit + st.outOfs, st.count, T, &sm.ring[lane][0]);
      }
      const unsigned okmask = __ballot_sync(gmask, good);
      if ((okmask & gmask) != gmask) ok = false;
    }
    if (sub == 0 && !ok) sliceUnits[w].huf_err = ZE_corruption_detected;           // :742
  }
}

// k_seq_blk : k_seq's mapping (one unit per lane, tables bank-interleaved), persistent over the launch's units
__global__ void __launch_bounds__(32) k_seq_blk(DecodeArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SeqSmem& sm = *reinterpret_cast<SeqSmem*>(smem_raw);
  const u32 lane = threadIdx.x;
  const u32 nunits = a.cnt[0];
  if (blockIdx.x * 32 >= nunits) return;
  if (lane < 3) {
    s16* norm = &sm.norm[0][lane]; u16* next = &sm.next[0][lane];
    Strided<s16> nv{norm, 32}; Strided<u16> sn{next, 32};
    if (lane == 0) { for (int i = 0; i < 36; i++) nv[i] = kLLnorm[i]; build_seq_table(sm.defLL, 1, nv, 35, 6, sn); }
    if (lane == 1) { for (int i = 0; i < 29; i++) nv[i] = kOFnorm[i]; build_seq_table(sm.defOF, 1, nv, 28, 5, sn); }
    if (lane == 2) { for (int i = 0; i < 53; i++) nv[i] = kMLnorm[i]; build_seq_table(sm.defML, 1, nv, 52, 6, sn); }
  }
  for (u32 i = lane; i < 36; i += 32) sm.llInfo[i] = ll_info(i);
  for (u32 i = lane; i < 53; i += 32) sm.mlInfo[i] = ml_info(i);
  __syncwarp();
  BlockUnit* const sliceUnits = a.units + unit_slice_base(a);
  for (u32 w = blockIdx.x * 32 + lane; w < nunits; w += gridDim.x * 32) {
    const BlockUnit u = sliceUnits[w];
    const u32 f = u.frame;
    const FrameInfo fi = a.info[f];
    SeqTableSet T;
    T.space[KIND_LL] = &sm.ll[0][lane]; T.space[KIND_ML] = &sm.ml[0][lane]; T.space[KIND_OF] = &sm.of[0][lane]; T.stride = 32;
    T.defs[KIND_LL] = sm.defLL; T.defs[KIND_OF] = sm.defOF; T.defs[KIND_ML] = sm.defML;
    UnitEmitter em;
    em.init(seq_region(a, f, fi) + u.rec_off, sm.llInfo, sm.mlInfo);
    seq_decode_unit(a.src_base + a.src_off[f], u, sliceUnits + fi.unit_base, fi.window, T, em, sm.llInfo, sm.mlInfo,
                    Strided<s16>{&sm.norm[0][lane], 32}, Strided<u16>{&sm.next[0][lane], 32}, &sm.ring[lane][0], a.dict);
    if (em.dead) { sliceUnits[w].seq_err_code = em.err_code; sliceUnits[w].seq_err_index = em.err_index; }
    else if (em.n) {
      sliceUnits[w].rep[0] = em.h.v0; sliceUnits[w].rep[1] = em.h.v1; sliceUnits[w].rep[2] = em.h.v2;
      sliceUnits[w].rep_sym = em.h.t0 | (em.h.t1 << 3) | (em.h.t2 << 6);
    }
  }
}

// k_exec_big : one CTA of W warps per FI_PAR frame.  The frame's work is cut into GROUPS in output order — 32 sequence
// records, a raw / RLE block, or a block's last literals — and group G belongs to warp G % W.  A warp that has written
// its group marks it in a small ring; whoever gets there moves the in-order chain (groups complete, watermark = output
// bytes that are final) over every consecutive written group.  Literal runs never wait; a match whose source lies
// before its group waits until the watermark has passed that source; sources inside the group are resolved in dependency
// rounds exactly as in k_exec.  So the record loads, the literal copies and the far-memory matches of up to W
// consecutive groups overlap, which one warp per large frame cannot do; what stays serial is the chain "group G-1
// complete -> the few matches of G that read its output -> G complete" (one L2 round trip per round: measured
// 1.8 us per group, DESIGN.md).  W follows from how many FI_PAR frames the launch holds (execb_warps): few large
// frames need the parallelism inside a frame, many frames fill the device on their own and a single warp each has no
// synchronisation cost.  All three instantiations are launched; the two that do not match return at once.
#ifndef EXECB_SLEEP
#define EXECB_SLEEP 100   // ns between two looks at the chain state while waiting (polling warps cost issue slots)
#endif
__host__ __device__ inline u32 execb_warps(u32 npar) { return npar <= 148 * 7 ? 4 : (npar <= 148 * 16 ? 2 : 1); }   // (7 CTAs of 4 + 1 warps per SM)
template <int W> struct ExecBigShared {
  volatile u32 wm;                // watermark: frame-relative output bytes that are final (every group before is complete)
  volatile u32 done;              // groups completed in order
  volatile u32 errG;              // lowest group that failed a record check (0xFFFFFFFF = none)
  volatile u32 flag[4 * W];       // flag[G % RING] == G + 1: group G has been written (RING = 4 W groups may be in flight)
  volatile u32 endPos[4 * W];
  u32 errAt[W], errCode[W];
  // W == 4 only: a fifth warp hashes the output behind the watermark (the content checksum of a long frame is a serial
  // chain of its own: done here it costs no time of its own, in k_xxh_big it did)
  volatile u32 left;              // worker warps that have finished the frame
  u32 hashed; u64 hv[4];          // bytes hashed and the four XXH64 accumulators when the hashing warp stops
};
// Group G (ending at output position endPos) has been written: mark it, then move the chain as far as it goes.
template <int W>
__device__ __forceinline__ void chain_publish(ExecBigShared<W>& sh, u32 G, u32 endPos, u32 lane) {
  __threadfence_block();
  __syncwarp();
  if (lane == 0) {
    if (W == 1) { sh.wm = endPos; sh.done = G + 1; }
    else {
      sh.endPos[G % (4 * W)] = endPos;
      __threadfence_block();
      sh.flag[G % (4 * W)] = G + 1;
      __threadfence_block();                                                       // (store flag, load done) vs (CAS done, load flag)
      u32 d = sh.done;
      while (sh.flag[d % (4 * W)] == d + 1) {
        const u32 e = sh.endPos[d % (4 * W)];
        if (atomicCAS((u32*)&sh.done, d, d + 1) == d) atomicMax((u32*)&sh.wm, e);
        __threadfence_block();
        d = sh.done;
      }
    }
  }
  __syncwarp();
}
// before group G starts: its ring slot must be free (group G - RING consumed by the chain); false = an earlier group failed
template <int W>
__device__ __forceinline__ bool chain_admit(ExecBigShared<W>& sh, u32 G, u32 lane) {
  if (W == 1) return true;
  u32 ok = 1;
  if (lane == 0) { while (G >= sh.done + 4 * W) { if (sh.errG < G) { ok = 0; break; } __nanosleep(EXECB_SLEEP); } }
  return __shfl_sync(FULLMASK, ok, 0) != 0;
}
// waits until the watermark has moved past `seen`; false = an earlier group failed
template <int W>
__device__ __forceinline__ bool chain_wait_move(ExecBigShared<W>& sh, u32 G, u32 seen, u32 lane) {
  u32 ok = 1;
  if (lane == 0) { while (sh.wm == seen) { if (sh.errG < G) { ok = 0; break; } __nanosleep(EXECB_SLEEP); } }
  return __shfl_sync(FULLMASK, ok, 0) != 0;
}

template <bool DICT, int W>
__global__ void __launch_bounds__((W + (W == 4)) * 32, W == 4 ? 7 : 32 / W) k_exec_big(DecodeArgs a) {
  __shared__ ExecBigShared<W> sh;
  constexpr bool HASH = W == 4;
  const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const u32 npar = a.cnt[1];
  if (execb_warps(npar) != (u32)W) return;
  const BlockUnit* const sliceUnits = a.units + unit_slice_base(a);
  for (u32 p = blockIdx.x; p < npar; p += gridDim.x) {
    __syncthreads();
    if (threadIdx.x == 0) { sh.wm = 0; sh.done = 0; sh.errG = 0xFFFFFFFFu; sh.left = 0; sh.hashed = 0; }
    if (threadIdx.x < (4 * W)) sh.flag[threadIdx.x] = 0;
    if (lane == 0 && warp < W) sh.errAt[warp] = 0xFFFFFFFFu;
    __syncthreads();
    const u32 f = a.par_list[a.item_base + p];
    const FrameInfo fi = a.info[f];
    const u8* src = a.src_base + a.src_off[f]; const u32 size = a.src_size[f];
    u8* dst = a.dst_base + frame_dst_off(a, f, fi); const u32 cap = frame_cap(a, f, fi);
    if (HASH && warp == W) {
      // ---- the hashing warp: XXH64 stripes of everything below the watermark (all lanes run the chain of accumulator
      //      lane & 3 on the same addresses; lanes 0-3 deliver) ----
      if (fi.flags & FI_CHECKSUM) {
        const u32 sub = lane & 3;
        u64 v = sub == 0 ? XP1 + XP2 : (sub == 1 ? XP2 : (sub == 2 ? 0 : 0 - XP1));
        const u8* q = dst + 8 * sub; u32 hashed = 0;
        while (true) {
          const u32 left = sh.left;                                                // before the watermark: all gone => it is final
          __threadfence_block();
          const u32 wmNow = __shfl_sync(FULLMASK, sh.wm, 0);
          __threadfence_block();
          u32 avail = (wmNow - hashed) >> 5;
          if (avail >= 8) {
            for (; avail >= 8; avail -= 8) {
              u64 x[8];
#pragma unroll
              for (int k = 0; k < 8; k++) x[k] = ldg64u(q + 32 * k);
#pragma unroll
              for (int k = 0; k < 8; k++) v = xxh_round(v, x[k]);
              q += 256; hashed += 256;
            }
            continue;
          }
          if (__shfl_sync(FULLMASK, left, 0) == (u32)W) {
            for (; avail; avail--) { v = xxh_round(v, ldg64u(q)); q += 32; hashed += 32; }
            break;
          }
          __nanosleep(4 * EXECB_SLEEP);
        }
        if (lane < 4) sh.hv[lane] = v;
        if (lane == 0) sh.hashed = hashed;
      }
      __syncthreads();
      continue;
    }
    const u8* litScratch = lit_region(a, f, fi);
    const SeqRec* recs = seq_region(a, f, fi);
    const BlockUnit* units = sliceUnits + fi.unit_base;
    u32 pos = fi.body_off, op = 0, G = 0, cblk = 0;
    bool litEntropy = false, bail = false; u32 err = 0;
    u32 R[3] = {1, 4, 8};                                                          // ZStdInternal.cs:111
    const u32 dictContent = DICT ? a.dict->contentSize : 0;
    const u8* const dictEnd = DICT ? a.dict_bytes + a.dict->contentOff + dictContent : nullptr;
    if (DICT && a.dict->hasEntropy) { litEntropy = true; R[0] = a.dict->rep[0]; R[1] = a.dict->rep[1]; R[2] = a.dict->rep[2]; }
    if (DICT && !a.dict->hasEntropy) { R[0] = a.dict->rep[0]; R[1] = a.dict->rep[1]; R[2] = a.dict->rep[2]; }
    while (true) {
      BlockHdr bh;
      err = read_block_hdr(src + pos, size - pos, bh);
      if (err) break;
      pos += 3;
      if (bh.type == 0) {                                                          // raw, :662-667
        if (bh.csize > cap - op) { err = ZE_dstSize_tooSmall; break; }
        if (G % W == warp) {
          if (!chain_admit(sh, G, lane)) { bail = true; break; }
          warp_copy(dst + op, src + pos, bh.csize, lane);
          chain_publish(sh, G, op + bh.csize, lane);
        }
        G++; op += bh.csize;
      } else if (bh.type == 1) {                                                   // RLE, :1945-1950
        if (bh.orig > cap - op) { err = ZE_dstSize_tooSmall; break; }
        if (G % W == warp) {
          if (!chain_admit(sh, G, lane)) { bail = true; break; }
          warp_fill(dst + op, src[pos], bh.orig, lane);
          chain_publish(sh, G, op + bh.orig, lane);
        }
        G++; op += bh.orig;
      } else {
        const BlockUnit bu = units[cblk]; cblk++;
        const u8* bp = src + pos; const u32 bsz = bh.csize;
        LitHdr lh; bool needs;
        read_lit_hdr(bp, bsz, lh, &needs);                                         // sound, and a needed table exists: par_walk
        const u8* lit; u32 rleByte = 0; bool isRle = false;
        if (lh.type >= 2) {
          if (bu.huf_err) { err = bu.huf_err; break; }                             // :742
          litEntropy = true; lit = litScratch + bu.lit_off;
        } else if (lh.type == 0) lit = bp + lh.lhSize;
        else { lit = nullptr; isRle = true; rleByte = bp[lh.lhSize]; }
        const u32 litSize = lh.litSize;
        const u8* sp = bp + lh.consumed; const u32 ssz = bsz - lh.consumed;
        u32 nbSeq, modes, hdr;
        read_seq_count(sp, ssz, &nbSeq, &modes, &hdr);
        if (bu.seq_err_code && bu.seq_err_index == 0xFFFFFFFFu) { err = bu.seq_err_code; break; }
        u32 litPos = 0;
        if (nbSeq) {
          const uint4 h = __ldg(reinterpret_cast<const uint4*>(recs + bu.rec_off));
          const u32 nRecs = h.x, outBytes = h.y, litBytes = h.z;
          const uint4* rv = reinterpret_cast<const uint4*>(recs + bu.rec_off + 1);
          const u32 blockBase = op;
          for (u32 g0 = 0; g0 < nRecs; g0 += 32, G++) {
            if (G % W != warp) continue;
            if (!chain_admit(sh, G, lane)) { bail = true; break; }
            const bool valid = g0 + lane < nRecs;
            const uint4 rec = valid ? __ldg(rv + g0 + lane) : make_uint4(0, 0, 0, 0);
            if (lane < 2 && g0 + 32 * W < nRecs) prefetch_line(rv + g0 + 32 * W + 16 * lane);   // this warp's next group
            const u32 ll = valid ? (rec.w & 0x1FFFF) : 0, ml = valid ? ((rec.w >> 17) | (((rec.y >> 18) & 7) << 15)) : 0, lpos = rec.y & 0x3FFFF;
            const u32 off = repsym_resolve(rec.z, (rec.y >> 21) & 7, R);
            const u64 start64 = (u64)blockBase + rec.x;
            const bool e1 = valid && start64 + ll + ml > cap;
            const bool e2 = valid && lpos + ll > litSize;
            const bool e3 = valid && (u64)off > start64 + ll + dictContent;         // :1290-1294
            const unsigned bad = __ballot_sync(FULLMASK, e1 | e2 | e3);
            if (bad) {
              const u32 first = (u32)__ffs(bad) - 1;
              const u32 code = __shfl_sync(FULLMASK, e1 ? (u32)ZE_dstSize_tooSmall : (u32)ZE_corruption_detected, first);
              if (lane == 0) { sh.errAt[warp] = G; sh.errCode[warp] = code; atomicMin((u32*)&sh.errG, G); }
              bail = true; break;
            }
            const u32 base = __shfl_sync(FULLMASK, rec.x, 0), lbase = __shfl_sync(FULLMASK, lpos, 0);
            const u32 gstart = blockBase + base;                                   // frame-relative output position of the group
            const u32 excl = valid ? rec.x - base : 0, mrel = excl + ll, incl = valid ? mrel + ml : 0xFFFFFFFFu;
            const u32 lsrc = lpos - lbase;
            u8* const g = dst + gstart;
            const u32 gend = gstart + __shfl_sync(FULLMASK, valid ? mrel + ml : 0, min(31u, nRecs - g0 - 1));
            // ---- literals ----
            {
              const bool bigL = ll >= 128;
              unsigned bigMask = __ballot_sync(FULLMASK, bigL);
              const u32 ls = bigL ? 0 : ll;
              const u32 lu = word_units(g + excl, ls);
              const u32 sincl = warp_incl_scan(lu, lane), sexcl = sincl - lu;
              const u32 Ls = __shfl_sync(FULLMASK, sincl, 31);
              if (isRle) { if (Ls) flat_fill_w<1>(g, rleByte * 0x01010101u, Ls, sincl, sexcl, excl, ls, lane); }
              else if (Ls > 32) flat_copy_w<2>(g, lit + lbase, Ls, sincl, sexcl, excl, lsrc, ls, lane);
              else if (Ls) flat_copy_w<1>(g, lit + lbase, Ls, sincl, sexcl, excl, lsrc, ls, lane);
              while (bigMask) {
                const u32 j = (u32)__ffs(bigMask) - 1; bigMask &= bigMask - 1;
                const u32 dj = __shfl_sync(FULLMASK, excl, j), nj = __shfl_sync(FULLMASK, ll, j), lj = __shfl_sync(FULLMASK, lsrc, j);
                if (isRle) warp_fill(g + dj, (u8)rleByte, nj, lane); else warp_copy(g + dj, lit + lbase + lj, nj, lane);
              }
            }
            __syncwarp();
            // ---- matches ----
            const bool hasM = ml > 0 && off != 0;
            const unsigned matchMask = __ballot_sync(FULLMASK, hasM);
            if (matchMask) {
              const i64 slo = (i64)mrel - (i64)off;                                // source range, group-relative
              // a source before the group needs the watermark to have passed it (<= 0: the dictionary, always there)
              u32 needAbs = 0;
              if (hasM && slo < 0) {
                const i64 endAbs = (i64)gstart + (slo + (i64)ml < 0 ? slo + (i64)ml : 0);
                needAbs = endAbs > 0 ? (u32)endAbs : 0;
              }
              unsigned depMask = 0;
              {
                i64 shi = slo + (i64)ml; if (shi > (i64)mrel) shi = (i64)mrel;
                const bool dep = hasM && shi > 0;
                const u32 needLo = slo > 0 ? (u32)slo : 0, needHi = dep ? (u32)shi : 1;
                const u32 aIdx = warp_upper_bound(incl, dep ? needLo : 0), bIdx = warp_upper_bound(incl, needHi - 1);
                if (dep) {
                  const unsigned upTo = bIdx >= 31 ? 0xFFFFFFFFu : ((1u << (bIdx + 1)) - 1);
                  depMask = upTo & ~((1u << aIdx) - 1) & ((1u << lane) - 1) & matchMask;
                }
              }
              unsigned doneMask = ~matchMask;
              while (doneMask != 0xFFFFFFFFu) {
                const u32 wmNow = __shfl_sync(FULLMASK, sh.wm, 0);
                __threadfence_block();
                const bool ready = hasM && !((doneMask >> lane) & 1) && ((depMask & ~doneMask) == 0) && needAbs <= wmNow;
                const unsigned Rdy = __ballot_sync(FULLMASK, ready);
                if (!Rdy) {                                                        // every pending match waits for earlier groups
                  if (!chain_wait_move(sh, G, wmNow, lane)) { bail = true; break; }
                  continue;
                }
                const bool inDict = DICT && off > gstart + mrel;
                const bool plain = ready && off >= ml && ml < 128 && !inDict;
                const u32 len = plain ? ml : 0, units4 = (len + 3) >> 2;
                const u32 pincl = warp_incl_scan(units4, lane), pexcl = pincl - units4;
                const u32 Tt = __shfl_sync(FULLMASK, pincl, 31);
                if (Tt > 32) flat_copy_m4<2>(g, Tt, pincl, pexcl, mrel, off, len, lane);
                else if (Tt) flat_copy_m4<1>(g, Tt, pincl, pexcl, mrel, off, len, lane);
                unsigned big = __ballot_sync(FULLMASK, ready && !plain);
                while (big) {
                  const u32 j = (u32)__ffs(big) - 1; big &= big - 1;
                  const u32 mj = __shfl_sync(FULLMASK, mrel, j), oj = __shfl_sync(FULLMASK, off, j), nj = __shfl_sync(FULLMASK, ml, j);
                  const u32 pj = gstart + mj;
                  if (DICT && oj > pj) {
                    const u32 back = oj - pj, l1 = back < nj ? back : nj;
                    warp_copy(g + mj, dictEnd - back, l1, lane);
                    __syncwarp();
                    if (nj > l1) warp_match(g + mj + l1, pj + l1, nj - l1, lane);
                  } else warp_match(g + mj, oj, nj, lane);
                }
                __syncwarp();
                doneMask |= Rdy;
              }
              if (bail) break;
            }
            chain_publish(sh, G, gend, lane);
          }
          if (bail) break;
          if (bu.seq_err_code) { err = bu.seq_err_code; break; }                   // :1594 after the decodable prefix
          op = blockBase + outBytes; litPos = litBytes;
          // the repeat offsets after this block, from its symbolic history (zb_blocks.cuh)
          const u32 n0 = repsym_resolve(bu.rep[0], bu.rep_sym & 7, R), n1 = repsym_resolve(bu.rep[1], (bu.rep_sym >> 3) & 7, R),
                    n2 = repsym_resolve(bu.rep[2], (bu.rep_sym >> 6) & 7, R);
          R[0] = n0; R[1] = n1; R[2] = n2;
        }
        // last literals (:1599-1605)
        const u32 lastLL = litSize - litPos;
        if (lastLL > cap - op) { err = ZE_dstSize_tooSmall; break; }
        if (G % W == warp) {
          if (!chain_admit(sh, G, lane)) { bail = true; break; }
          if (isRle) warp_fill(dst + op, (u8)rleByte, lastLL, lane); else warp_copy(dst + op, lit + litPos, lastLL, lane);
          chain_publish(sh, G, op + lastLL, lane);
        }
        G++; op += lastLL;
      }
      pos += bh.csize;
      if (bh.last) break;
    }
    if (HASH) { __threadfence_block(); __syncwarp(); if (lane == 0) atomicAdd((u32*)&sh.left, 1u); }
    __syncthreads();
    if (warp != 0) continue;
    // a failed record check comes before anything the warps met afterwards; without one, no warp left early and all
    // of them hold the same err / op / pos
    if (sh.errG != 0xFFFFFFFFu) {
      const u32 eg = sh.errG;
      for (u32 k = 0; k < W; k++) if (sh.errAt[k] == eg) err = sh.errCode[k];
    }
    // ---- frame epilogue (:2069-2085) and the multi-frame loop tail (:2111-2157), as k_exec ----
    bool needXxh = false; u32 trailer = 0;
    if (!err) {
      if ((fi.flags & FI_FCS_KNOWN) && op != fi.fcs) err = ZE_corruption_detected;
      else if (fi.flags & FI_CHECKSUM) {
        if (size - pos < 4) err = ZE_checksum_wrong; else { trailer = pos; pos += 4; needXxh = true; }
      }
    }
    u32 tailErr = 0, nextOff = 0;
    if (!err) {
      while (true) {
        u32 rem = size - pos;
        if (rem < 5) { if (rem) tailErr = ZE_srcSize_wrong; break; }
        u32 magic = ld32(src + pos);
        if (magic == MAGIC) { nextOff = pos; break; }
        if ((magic & 0xFFFFFFF0u) != MAGIC_SKIP) { tailErr = ZE_prefix_unknown; break; }
        if (rem < 8) { tailErr = ZE_srcSize_wrong; break; }
        u32 skip = ld32(src + pos + 4) + 8u;
        if (rem < skip) { tailErr = ZE_srcSize_wrong; break; }
        pos += skip;
      }
    }
    if (lane == 0) {
      u32 res = err ? zerr(err) : (tailErr ? zerr(tailErr) : fi.out_base + (u32)op);
      if (HASH && needXxh && sh.hashed == (op & ~31u)) {
        // the hashing warp has covered every stripe: finish the digest here (:2078-2082; k_xxh_big then skips the frame)
        const u64 h = xxh64_finish(sh.hv[0], sh.hv[1], sh.hv[2], sh.hv[3], dst, op);
        if ((u32)h != ld32(src + trailer)) res = zerr(ZE_checksum_wrong);
        needXxh = false;
      }
      a.result[f] = res;
      a.info[f].trailer_off = trailer; a.info[f].decoded = (u32)op; a.info[f].next_off = nextOff;
      a.info[f].flags = fi.flags | (needXxh ? FI_NEED_XXH : 0);
      if (nextOff && a.more) atomicAdd(a.more, 1u);
    }
  }
}

// =================================================================================================
// k_xxh : XXH64(seed 0) of the decoded bytes, 4 lanes per frame (one accumulator each)
// =================================================================================================
__global__ void __launch_bounds__(128) k_xxh(DecodeArgs a) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 f = t >> 2, sub = t & 3, lane = threadIdx.x & 31;
  const unsigned gmask = 0xFu << (lane & ~3u);
  if (f >= a.n) return;
  FrameInfo fi = a.info[f];
  if (!(fi.flags & FI_NEED_XXH) || (fi.flags & FI_PAR)) return;
  const u8* dst = a.dst_base + frame_dst_off(a, f, fi);
  u64 h = xxh64_group<false>(dst, fi.decoded, sub, gmask, lane & ~3u);
  if (sub == 0) {
    const u8* src = a.src_base + a.src_off[f];
    if ((u32)h != ld32(src + fi.trailer_off)) a.result[f] = zerr(ZE_checksum_wrong);   // :2078-2082
  }
}
// the FI_PAR frames (few and long): the same 4 lanes per frame with the deeper load pipeline, persistent over the list
__global__ void __launch_bounds__(32) k_xxh_big(DecodeArgs a) {
  const u32 lane = threadIdx.x, sub = lane & 3, slot = lane >> 2;
  const unsigned gmask = 0xFu << (lane & ~3u);
  const u32 npar = a.cnt[1];
  for (u32 p = blockIdx.x * 8 + slot; p < npar; p += gridDim.x * 8) {
    const u32 f = a.par_list[a.item_base + p];
    const FrameInfo fi = a.info[f];
    if (!(fi.flags & FI_NEED_XXH)) continue;
    const u8* dst = a.dst_base + frame_dst_off(a, f, fi);
    const u64 h = xxh64_group<true>(dst, fi.decoded, sub, gmask, lane & ~3u);
    if (sub == 0) {
      const u8* src = a.src_base + a.src_off[f];
      if ((u32)h != ld32(src + fi.trailer_off)) a.result[f] = zerr(ZE_checksum_wrong);
    }
  }
}


// =================================================================================================
// launch
// =================================================================================================
size_t decode_lit_arena_bytes(u64 max_dst_bytes, u64 max_items) { return (size_t)(max_dst_bytes + 64 * (max_items + 2) + 256); }
size_t decode_seq_arena_bytes(u64 max_dst_bytes, u64 max_items) { return (size_t)((2 * (max_dst_bytes / 3) + 32 * (max_items + 2) + 64) * sizeof(SeqRec)); }

// k_dict : one thread parses the context's dictionary into a DictState (zb_format.cuh dict_load)
__global__ void __launch_bounds__(32) k_dict(const u8* dict, u32 size, DictState* ds) {
  __shared__ HufBuildWk wk; __shared__ HufFseScratch fs; __shared__ u8 slot[260]; __shared__ s16 norm[64]; __shared__ u16 next[64];
  if (threadIdx.x == 0) dict_load(dict, size, *ds, wk, fs, slot, norm, next);
}
cudaError_t decode_load_dictionary(const u8* d_dict_bytes, u32 size, DictState* d_state, cudaStream_t st) {
  k_dict<<<1, 32, 0, st>>>(d_dict_bytes, size, d_state);
  return cudaGetLastError();
}

// grids of the persistent block-parallel kernels: what one wave of the device holds (set by decode_configure)
static int g_par_grid_huf = 148 * 5, g_grid_huf_small = 148 * 11, g_par_grid_seq = 148 * 2, g_par_grid_exec = 148 * 32;   // (exec: in warps)
int decode_huf_ctas() { return g_grid_huf_small > g_par_grid_huf ? g_grid_huf_small : g_par_grid_huf; }
size_t decode_unit_arena_count(u64 max_dst_bytes, u64 max_items) { return (size_t)(max_dst_bytes / PAR_UNIT_BYTES + PAR_UNIT_SLACK * (max_items + 2) + 64); }

cudaError_t decode_configure() {
  cudaError_t e = cudaFuncSetAttribute(k_huf<HUF_TABLE_LOG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HufSmem<HUF_TABLE_LOG>));
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(k_huf<HUF_ROOT_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HufSmem<HUF_ROOT_SMALL>));
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(k_huf_blk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HufSmem<HUF_TABLE_LOG>));
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(k_seq_blk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SeqSmem));
  if (e != cudaSuccess) return e;
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) {
    int per = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_huf_blk, 32, sizeof(HufSmem<HUF_TABLE_LOG>)) == cudaSuccess && per > 0) g_par_grid_huf = sms * per;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_huf<HUF_ROOT_SMALL>, 32, sizeof(HufSmem<HUF_ROOT_SMALL>)) == cudaSuccess && per > 0) g_grid_huf_small = sms * per;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_seq_blk, 32, sizeof(SeqSmem)) == cudaSuccess && per > 0) g_par_grid_seq = sms * per;
    g_par_grid_exec = sms * 32;
  }
  e = cudaFuncSetAttribute(k_seq_t<2, 8, 8, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SeqSmemT<8, 8, 8>));
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(k_seq_t<0, 9, 8, 9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SeqSmem));
}

const char* const kDecodeKernelNames[DECODE_KERNELS] = {"k_parse", "k_huf", "k_seq", "k_exec", "k_xxh"};

// The whole pipeline on one stream.  Running the entropy stages of one slice beside the execute stages of another on a
// second stream measured slower (the execute warps starve the lone FSE warps of an SM).
cudaError_t decode_launch(const DecodeArgs& a, cudaStream_t st, int* launches, cudaEvent_t* marks) {
  if (a.n == 0) return cudaSuccess;
  { cudaError_t e = cudaMemsetAsync(a.cnt, 0, 32, st); if (e != cudaSuccess) return e; }
  if (marks) cudaEventRecord(marks[0], st);
  k_parse<<<(a.n + 127) / 128, 128, 0, st>>>(a);
  if (marks) cudaEventRecord(marks[1], st);
  { const u32 need = (a.n + 7) / 8;
    k_huf<HUF_ROOT_SMALL><<<need < (u32)g_grid_huf_small ? need : (u32)g_grid_huf_small, 32, sizeof(HufSmem<HUF_ROOT_SMALL>), st>>>(a);
    k_huf<HUF_TABLE_LOG><<<need < (u32)g_par_grid_huf ? need : (u32)g_par_grid_huf, 32, sizeof(HufSmem<HUF_TABLE_LOG>), st>>>(a); }
  if (a.units) k_huf_blk<<<g_par_grid_huf, 32, sizeof(HufSmem<HUF_TABLE_LOG>), st>>>(a);
  if (marks) cudaEventRecord(marks[2], st);
  k_seq_t<1, 6, 6, 7><<<(a.n + 31) / 32, 32, sizeof(SeqSmemT<6, 6, 7>), st>>>(a);
  k_seq_t<2, 8, 8, 8><<<(a.n + 31) / 32, 32, sizeof(SeqSmemT<8, 8, 8>), st>>>(a);
  k_seq_t<0, 9, 8, 9><<<(a.n + 31) / 32, 32, sizeof(SeqSmem), st>>>(a);
  if (a.units) k_seq_blk<<<g_par_grid_seq, 32, sizeof(SeqSmem), st>>>(a);
  if (marks) cudaEventRecord(marks[3], st);
  if (launches) *launches += a.units ? 8 : 6;
  { cudaError_t e = cudaGetLastError(); if (e != cudaSuccess) return e; }
  if (a.dict) k_exec<true><<<(a.n + (EXEC_THREADS / 32) - 1) / (EXEC_THREADS / 32), EXEC_THREADS, 0, st>>>(a);
  else k_exec<false><<<(a.n + (EXEC_THREADS / 32) - 1) / (EXEC_THREADS / 32), EXEC_THREADS, 0, st>>>(a);
  if (a.units) {
    if (a.dict) {
      k_exec_big<true, 4><<<g_par_grid_exec / 32 * 7, 160, 0, st>>>(a); k_exec_big<true, 2><<<g_par_grid_exec / 2, 64, 0, st>>>(a); k_exec_big<true, 1><<<g_par_grid_exec, 32, 0, st>>>(a);
    } else {
      k_exec_big<false, 4><<<g_par_grid_exec / 32 * 7, 160, 0, st>>>(a); k_exec_big<false, 2><<<g_par_grid_exec / 2, 64, 0, st>>>(a); k_exec_big<false, 1><<<g_par_grid_exec, 32, 0, st>>>(a);
    }
  }
  if (marks) cudaEventRecord(marks[4], st);
  k_xxh<<<(a.n * 4 + 127) / 128, 128, 0, st>>>(a);
  if (a.units) k_xxh_big<<<148 * 8, 32, 0, st>>>(a);
  if (marks) cudaEventRecord(marks[5], st);
  if (launches) *launches += a.units ? 6 : 2;
  return cudaGetLastError();
}

}  // namespace zb
