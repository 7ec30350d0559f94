// zb_exec_copy.cuh — the execute stage's flattened copies: the short literal runs, RLE fills and non-overlapping matches of
// one group of 32 sequences, moved by the whole warp at once (k_exec, k_exec_big; tests/gpu_harness/exec_copy.cu).
//
// Each lane's run is cut into units, U rows of 32 units are in flight per pass, and a lane finds the run of its unit with
// a shuffle binary search over the inclusive prefix sums of the units per run.  A store never writes a byte outside its
// own run: the other bytes of a word may belong to another lane's run of the same pass, to a match that is written in a
// later round, or to the neighbouring frame of another warp.
#pragma once
#include "zb_common.cuh"

#ifndef FULLMASK
#define FULLMASK 0xFFFFFFFFu
#endif

namespace zb {

__device__ __forceinline__ u32 warp_incl_scan(u32 v, u32 lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { u32 t = __shfl_up_sync(0xFFFFFFFFu, v, d); if (lane >= (u32)d) v += t; }
  return v;
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

// the short literal runs of a group (ls = 0 for the others), flattened over the lanes
__device__ __forceinline__ void flat_literals(u8* g, const u8* lit, bool isRle, u32 rleByte, u32 excl, u32 lsrc, u32 ls, u32 lane) {
  const u32 lu = word_units(g + excl, ls);
  const u32 sincl = warp_incl_scan(lu, lane), sexcl = sincl - lu;
  const u32 Ls = __shfl_sync(FULLMASK, sincl, 31);
  if (isRle) { if (Ls) flat_fill_w<1>(g, rleByte * 0x01010101u, Ls, sincl, sexcl, excl, ls, lane); }
  else if (Ls > 32) flat_copy_w<2>(g, lit, Ls, sincl, sexcl, excl, lsrc, ls, lane);
  else if (Ls) flat_copy_w<1>(g, lit, Ls, sincl, sexcl, excl, lsrc, ls, lane);
}
// the short non-overlapping matches of a round (len = 0 for the others), flattened over the lanes.  (Measured slower in
// 8-byte units, destination-aligned or source-relative: DESIGN.md §7.)
__device__ __forceinline__ void flat_matches(u8* g, u32 mrel, u32 off, u32 len, u32 lane) {
  const u32 units = (len + 3) >> 2;
  const u32 pincl = warp_incl_scan(units, lane), pexcl = pincl - units;
  const u32 Tt = __shfl_sync(FULLMASK, pincl, 31);
  if (Tt > 32) flat_copy_m4<2>(g, Tt, pincl, pexcl, mrel, off, len, lane);
  else if (Tt) flat_copy_m4<1>(g, Tt, pincl, pexcl, mrel, off, len, lane);
}

}  // namespace zb
