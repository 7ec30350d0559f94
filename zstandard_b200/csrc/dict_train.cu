// dict_train.cu — sm_100a kernels and host driver of zstdb200_train_dictionary (fastCover selection, zb_dict_train.cuh).
//
//   k_dt_hash    : thread / position   the d-mer hash of every training position
//   k_dt_prev    : CTA / 2048 positions the last earlier position with the same hash within DT_LOOKBACK (bitonic sort of
//                                      (hash, position) keys of the tile and the DT_LOOKBACK positions before it in shared memory)
//   k_dt_freq    : warp / sample       the frequency pass (global atomics)
//   k_dt_select  : CTA / candidate k   the epochs, one after another: every position adds its frequency to the window ends
//                                      it is the first occurrence of its hash in (difference array), a prefix scan gives every
//                                      window's score, a first-max reduction the serial loop's choice; then the chosen
//                                      window's frequencies are zeroed and its bytes copied
// The entropy statistics come from the encoder's match stage (encode_match_stats) and the tables from zb_dict_train.cuh on
// the host; search candidates are scored with the dictionary encoder (encode_launch).
#include <cuda_runtime.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>

#include "dict_train.cuh"
#include "encode_kernels.cuh"
#include "zb_dict_train.cuh"

namespace zb {

static_assert(sizeof(DtStats) == DT_STAT_WORDS * 4, "k_enc_stats writes DtStats");
static constexpr u32 kNone = 0xFFFFFFFFu;
static constexpr u32 kPrevTile = 2048;

__global__ void k_dt_hash(const u8* samples, u32 nbDmers, u32 f, u32 d, u32* hash) {
  for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < nbDmers; j += gridDim.x * blockDim.x) hash[j] = dt_hash(samples + j, f, d);
}

// prev[j] for j in the CTA's tile [s, s + kPrevTile): the last j' in [s - DT_LOOKBACK, j) with hash[j'] == hash[j], or kNone.
// Any j' within L - 1 <= DT_LOOKBACK - 1 positions of j is found, which is all the scoring needs.
__global__ void __launch_bounds__(1024) k_dt_prev(const u32* hash, u32 nbDmers, u32* prev) {
  constexpr u32 N = kPrevTile + DT_LOOKBACK;
  __shared__ u64 key[N];
  const u32 s = blockIdx.x * kPrevTile, lo = s >= DT_LOOKBACK ? s - DT_LOOKBACK : 0;
  for (u32 i = threadIdx.x; i < N; i += blockDim.x) {
    const u32 j = lo + i;
    key[i] = j < nbDmers && j < s + kPrevTile ? ((u64)hash[j] << 32) | j : ~0ull;
  }
  __syncthreads();
  for (u32 size = 2; size <= N; size <<= 1)
    for (u32 stride = size >> 1; stride > 0; stride >>= 1) {
      for (u32 t = threadIdx.x; t < N / 2; t += blockDim.x) {
        const u32 i = 2 * t - (t & (stride - 1)), k = i + stride;
        const bool up = (i & size) == 0;
        const u64 a = key[i], b = key[k];
        if ((a > b) == up) { key[i] = b; key[k] = a; }
      }
      __syncthreads();
    }
  for (u32 i = threadIdx.x; i < N; i += blockDim.x) {
    const u64 v = key[i];
    const u32 j = (u32)v;
    if (v == ~0ull || j < s) continue;
    prev[j] = i > 0 && (key[i - 1] >> 32) == (v >> 32) ? (u32)key[i - 1] : kNone;
  }
}

// FASTCOVER_computeFrequency: one warp per training sample
__global__ void k_dt_freq(const u64* off, u32 nbTrain, u32 readLen, u32 skip, const u32* hash, u32* freqs) {
  const u32 lane = threadIdx.x & 31, nw = gridDim.x * (blockDim.x >> 5);
  for (u32 i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < nbTrain; i += nw) {
    const u64 b = off[i], e = off[i + 1];
    for (u64 p = b + (u64)lane * (skip + 1); p + readLen <= e; p += 32ull * (skip + 1)) atomicAdd(&freqs[hash[p]], 1u);
  }
}

struct DtSelectArgs {
  const u8* samples; const u32* hash; const u32* prev;
  u32 nbDmers, d, capacity;
  u32 k[DT_SEARCH_KS];
  u32* freqs[DT_SEARCH_KS]; u32* diff[DT_SEARCH_KS]; u8* sel[DT_SEARCH_KS];
  u32* tail;   // [DT_SEARCH_KS] out: where each selection starts in sel[c][0..capacity)
};

// One CTA per candidate.  Window W(t) = [max(b, t - L), t), t in (b, e]; position j is the first occurrence of its hash in W(t)
// for t in (max(j, prev_j + L), min(j + L, e)] when prev_j >= b, else for t in (j, min(j + L, e)]: it adds freqs[hash_j] there.
__global__ void __launch_bounds__(1024) k_dt_select(DtSelectArgs a) {
  __shared__ u32 wmaxv[32], wmaxt[32];
  __shared__ u32 sh_tail, sh_zero, sh_done, sh_best, sh_bestT;
  __shared__ u32 chunkSum[1024];
  const u32 c = blockIdx.x, tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5;
  const u32 k = a.k[c], d = a.d, L = k - d + 1;
  u32* const freqs = a.freqs[c]; u32* const diff = a.diff[c]; u8* const sel = a.sel[c];
  const DtEpochs ep = dt_epochs(a.capacity, a.nbDmers, k);
  if (tid == 0) { sh_tail = a.capacity; sh_zero = 0; sh_done = ep.num == 0; }
  __syncthreads();
  for (u32 epoch = 0; !sh_done; epoch = (epoch + 1) % ep.num) {
    const u32 b = epoch * ep.size, e = b + ep.size, n = ep.size;   // scores of t = b + 1 .. e at diff[1 .. n]
    for (u32 i = tid; i < n + 2; i += nt) diff[i] = 0;
    __syncthreads();
    for (u32 j = b + tid; j < e; j += nt) {
      const u32 v = freqs[a.hash[j]];
      if (!v) continue;
      const u32 pv = a.prev[j];
      const u32 lo = pv != kNone && pv >= b && pv + L > j ? pv + L : j, hi = j + L < e ? j + L : e;
      if (lo < hi) { atomicAdd(&diff[lo + 1 - b], v); atomicAdd(&diff[hi + 1 - b], 0u - v); }
    }
    __syncthreads();
    // prefix scan of diff[1..n] in nt contiguous chunks, then the first maximum
    const u32 per = (n + nt - 1) / nt, c0 = 1 + tid * per, c1 = min(c0 + per, n + 1);
    u32 sum = 0;
    for (u32 i = c0; i < c1; i++) sum += diff[i];
    chunkSum[tid] = sum;
    __syncthreads();
    if (wid == 0) {   // exclusive scan of the chunk sums by warp 0
      u32 carry = 0;
      for (u32 base = 0; base < nt; base += 32) {
        const u32 x = chunkSum[base + lane];
        u32 v = x;
        for (int o = 1; o < 32; o <<= 1) { const u32 y = __shfl_up_sync(0xFFFFFFFFu, v, o); if (lane >= (u32)o) v += y; }
        chunkSum[base + lane] = carry + v - x;
        carry += __shfl_sync(0xFFFFFFFFu, v, 31);
      }
    }
    __syncthreads();
    u32 run = chunkSum[tid], bestV = 0, bestT = kNone;
    for (u32 i = c0; i < c1; i++) { run += diff[i]; if (run > bestV) { bestV = run; bestT = b + i; } }
    for (int o = 16; o > 0; o >>= 1) {
      const u32 ov = __shfl_down_sync(0xFFFFFFFFu, bestV, o), ot = __shfl_down_sync(0xFFFFFFFFu, bestT, o);
      if (ov > bestV || (ov == bestV && ot < bestT)) { bestV = ov; bestT = ot; }
    }
    if (lane == 0) { wmaxv[wid] = bestV; wmaxt[wid] = bestT; }
    __syncthreads();
    if (tid == 0) {
      u32 bv = 0, bt = kNone;
      for (u32 w = 0; w < nt / 32; w++) if (wmaxv[w] > bv || (wmaxv[w] == bv && wmaxt[w] < bt)) { bv = wmaxv[w]; bt = wmaxt[w]; }
      sh_best = bv; sh_bestT = bt;
    }
    __syncthreads();
    if (sh_best == 0) {
      if (tid == 0 && ++sh_zero >= DT_ZERO_SCORE_RUN) sh_done = 1;
      __syncthreads();
      continue;
    }
    const u32 t = sh_bestT, sb = t - b > L ? t - L : b;
    const u32 len = min(t - sb + d - 1, sh_tail);
    for (u32 j = sb + tid; j < t; j += nt) freqs[a.hash[j]] = 0;
    __syncthreads();
    if (len < d) { if (tid == 0) sh_done = 1; __syncthreads(); break; }
    const u32 tail = sh_tail - len;
    for (u32 i = tid; i < len; i += nt) sel[tail + i] = a.samples[sb + i];
    __syncthreads();
    if (tid == 0) { sh_zero = 0; sh_tail = tail; if (tail == 0) sh_done = 1; }
    __syncthreads();
  }
  if (tid == 0) a.tail[c] = sh_tail;
}

namespace {

// device allocations of one training call, freed on every return path
struct DevBufs {
  std::vector<void*> p;
  ~DevBufs() { for (void* x : p) cudaFree(x); }
  template <class T> cudaError_t get(T** out, size_t bytes) {
    void* x = nullptr; cudaError_t e = cudaMalloc(&x, bytes ? bytes : 1);
    if (e == cudaSuccess) p.push_back(x);
    *out = (T*)x; return e;
  }
};

}  // namespace

#define DTCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(e_); return zerr(ZE_GENERIC); } } while (0)

u32 dt_train_run(DtDevice& dv, u8* dict, u32 capacity, const u8* samples, const u32* sizes, size_t n, zstdb200_train_params& pr, std::string& err) {
  const u32 k0 = pr.k, d = pr.d ? pr.d : 8, f = pr.f ? pr.f : 20, accel = pr.accel ? pr.accel : 1;
  const int level = pr.level ? pr.level : 3;
  if (d != 6 && d != 8) { err = "d must be 6 or 8"; return zerr(ZE_GENERIC); }
  if (f > DT_MAX_F) { err = "f must be at most 24"; return zerr(ZE_GENERIC); }
  if (accel > 10) { err = "accel must be 1..10"; return zerr(ZE_GENERIC); }
  if (pr.split_percent > 100) { err = "split_percent must be 1..100"; return zerr(ZE_GENERIC); }
  if (level < 1 || level > 3) { err = "level must be 1..3"; return zerr(ZE_GENERIC); }
  if (k0 && (k0 < d || k0 > DT_MAX_K)) { err = "k must be d..2048"; return zerr(ZE_GENERIC); }
  if (!samples && n) { err = "null samples"; return zerr(ZE_GENERIC); }
  const u32 split = pr.split_percent ? pr.split_percent : (k0 ? 100 : 75);
  if (capacity < DT_DICT_MIN || capacity < (k0 ? k0 : dt_search_k(DT_SEARCH_KS - 1))) return zerr(ZE_dstSize_tooSmall);
  std::vector<u64> off(n + 1, 0);
  for (size_t i = 0; i < n; i++) off[i + 1] = off[i] + sizes[i];
  const u64 total = off[n];
  if (total > 0xFFFFFFFFull) { err = "the samples total 2^32 bytes or more"; return zerr(ZE_GENERIC); }
  // ZDICT's conditions (FASTCOVER_ctx_init): the split is floor(n * split / 100) as ZDICT computes it from a double
  const u32 nbTrain = split < 100 ? (u32)((double)n * ((double)split / 100.0)) : (u32)n;
  const u32 nbTest = split < 100 ? (u32)n - nbTrain : 0;
  const u32 readLen = d > 8 ? d : 8;
  if (total < readLen || nbTrain < 5 || (!k0 && nbTest < 1)) return zerr(ZE_srcSize_wrong);
  if (off[nbTrain] < readLen) return zerr(ZE_srcSize_wrong);   // (ZDICT does not guard this: training bytes shorter than one d-mer)
  const u32 nbDmers = (u32)(off[nbTrain] - readLen + 1);
  const u32 nc = k0 ? 1 : DT_SEARCH_KS;
  cudaStream_t st = dv.stream;
  DevBufs mem;
  u8* dSamples; u64* dOff; u32 *dHash, *dPrev, *dFreq0, *dTail, *dStats;
  DTCK(mem.get(&dSamples, total + 64));
  DTCK(cudaMemcpyAsync(dSamples, samples, total, cudaMemcpyHostToDevice, st));
  DTCK(cudaMemsetAsync(dSamples + total, 0, 64, st));
  DTCK(mem.get(&dOff, (n + 1) * 8));
  DTCK(cudaMemcpyAsync(dOff, off.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
  DTCK(mem.get(&dHash, (size_t)nbDmers * 4));
  DTCK(mem.get(&dPrev, (size_t)nbDmers * 4));
  DTCK(mem.get(&dFreq0, (size_t)4 << f));
  DTCK(mem.get(&dTail, DT_SEARCH_KS * 4));
  DTCK(mem.get(&dStats, sizeof(DtStats)));
  DTCK(cudaMemsetAsync(dFreq0, 0, (size_t)4 << f, st));
  k_dt_hash<<<std::min<u32>((nbDmers + 255) / 256, 148 * 64), 256, 0, st>>>(dSamples, nbDmers, f, d, dHash);
  k_dt_prev<<<(nbDmers + kPrevTile - 1) / kPrevTile, 1024, 0, st>>>(dHash, nbDmers, dPrev);
  k_dt_freq<<<std::min<u32>((nbTrain + 7) / 8, 148 * 32), 256, 0, st>>>(dOff, nbTrain, readLen, dt_accel_skip(accel), dHash, dFreq0);
  dv.launches += 3;
  DtSelectArgs sa{};
  sa.samples = dSamples; sa.hash = dHash; sa.prev = dPrev; sa.nbDmers = nbDmers; sa.d = d; sa.capacity = capacity; sa.tail = dTail;
  for (u32 c = 0; c < nc; c++) {
    sa.k[c] = k0 ? k0 : dt_search_k(c);
    const DtEpochs ep = dt_epochs(capacity, nbDmers, sa.k[c]);
    DTCK(mem.get(&sa.freqs[c], (size_t)4 << f));
    DTCK(mem.get(&sa.diff[c], ((size_t)ep.size + 2) * 4));
    DTCK(mem.get(&sa.sel[c], capacity));
    DTCK(cudaMemcpyAsync(sa.freqs[c], dFreq0, (size_t)4 << f, cudaMemcpyDeviceToDevice, st));
  }
  k_dt_select<<<nc, 1024, 0, st>>>(sa);
  dv.launches += 1;
  DTCK(cudaGetLastError());
  u32 tails[DT_SEARCH_KS];
  std::vector<std::vector<u8>> sels(nc);
  DTCK(cudaMemcpyAsync(tails, dTail, nc * 4, cudaMemcpyDeviceToHost, st));
  DTCK(cudaStreamSynchronize(st));
  for (u32 c = 0; c < nc; c++) {
    sels[c].resize(capacity - tails[c]);
    DTCK(cudaMemcpyAsync(sels[c].data(), sa.sel[c] + tails[c], capacity - tails[c], cudaMemcpyDeviceToHost, st));
  }
  DTCK(cudaStreamSynchronize(st));

  // encoder dictionaries: host preparation as in zstdb200_load_dictionary, one device block reused by every candidate
  u8* dEnc = nullptr; size_t encCap = 0;
  std::vector<uint4> enc;
  auto upload = [&](const u8* bytes, u32 size, bool raw) -> cudaError_t {
    DictState ds;
    if (raw) dt_raw_dict_state(ds, size); else dict_load_host(bytes, size, ds);
    enc = enc_dict_block(bytes, size, ds);
    const size_t bytesNeeded = enc.size() * sizeof(uint4);
    if (bytesNeeded > encCap) { cudaError_t e = mem.get(&dEnc, bytesNeeded); if (e) return e; encCap = bytesNeeded; }
    cudaError_t e = cudaMemcpyAsync(dEnc, enc.data(), bytesNeeded, cudaMemcpyHostToDevice, st);
    if (e) return e;
    return cudaStreamSynchronize(st);   // enc is reused by the next upload
  };
  // sub-batches of [lo, hi) whose items (at offsets off[i] - off[lo], itemSize(i) bytes) fit the encoder's arenas
  auto cut = [&](u32 lo, u32 hi, auto itemSize, auto outBytes, std::vector<std::pair<u32, u32>>& subs) -> bool {
    subs.clear();
    u32 a = lo;
    while (a < hi) {
      u32 b = a; size_t out = 0;
      while (b < hi && b - a < dv.maxItems && off[b] - off[a] + itemSize(b) <= dv.maxBatch && out + outBytes(b) <= dv.dstCap) { out += outBytes(b); b++; }
      if (b == a) return false;
      subs.push_back({a, b}); a = b;
    }
    return true;
  };
  const u32 nFinal = (u32)((u64)nbTrain * dt_accel_finalize(accel) / 100);
  std::vector<std::pair<u32, u32>> finalSubs, testSubs;
  auto firstBlock = [&](u32 i) -> size_t { return std::min<u32>(sizes[i], BLOCKSIZE_MAX); };
  if (!cut(0, nFinal, firstBlock, [](u32) { return (size_t)0; }, finalSubs)) { err = "a sample does not fit max_batch_bytes"; return zerr(ZE_GENERIC); }
  u32 testMax = 0;
  for (u32 i = nbTrain; i < n; i++) testMax = std::max(testMax, sizes[i]);
  if (!k0 && !cut(nbTrain, (u32)n, [&](u32 i) { return (size_t)sizes[i]; }, [&](u32 i) { return align_up(encode_bound(sizes[i]), 16); }, testSubs)) {
    err = "a test sample is larger than the context's max_batch_bytes"; return zerr(ZE_GENERIC);
  }
  std::vector<u8> out(capacity), best;
  u64 bestScore = ~0ull; u32 bestK = 0;
  for (u32 c = 0; c < nc; c++) {
    const u32 selSize = (u32)sels[c].size();
    // entropy statistics: the match stage over the first block of each finalize sample against the raw selection
    DTCK(upload(sels[c].data(), selSize, true));
    DTCK(cudaMemsetAsync(dStats, 0, sizeof(DtStats), st));
    for (auto& sb : finalSubs) {
      const u32 m = sb.second - sb.first;
      const DescView h(dv.h_desc, m);   // no destinations: dstOff / dstCap are left as they are and not read
      u32 mx = 0;
      for (u32 q = 0; q < m; q++) { h.srcOff[q] = off[sb.first + q] - off[sb.first]; h.srcSize[q] = (u32)firstBlock(sb.first + q); mx = std::max(mx, h.srcSize[q]); }
      DTCK(cudaMemcpyAsync(dv.d_desc, dv.h_desc, DescView::bytes(m), cudaMemcpyHostToDevice, st));
      const Items it = DescView(dv.d_desc, m).items(dSamples + off[sb.first], nullptr, nullptr);
      int nl = 0;
      DTCK(encode_match_stats(encode_args(it, m, 0, level, 0, mx, ENC_EXCLUSIVE, dEnc, &enc), *dv.enc, st, dStats, &nl));
      dv.launches += nl;
      DTCK(cudaStreamSynchronize(st));   // the descriptors' pinned staging is rewritten by the next sub-batch
    }
    DtStats stats;
    DTCK(cudaMemcpyAsync(&stats, dStats, sizeof stats, cudaMemcpyDeviceToHost, st));
    DTCK(cudaStreamSynchronize(st));
    DtHeaderScratch hw; u8 hdr[DT_DICT_MIN];
    const u32 h = dt_write_header(hdr, pr.dict_id ? pr.dict_id : dt_dict_id(sels[c].data(), selSize), stats, selSize, hw);
    if (!h) { err = "entropy tables could not be written"; return zerr(ZE_GENERIC); }
    const u32 size = dt_assemble(out.data(), capacity, hdr, h, sels[c].data(), selSize);
    u64 score = 0;
    if (!k0) {   // compress the test samples with the finished dictionary
      DTCK(upload(out.data(), size, false));
      for (auto& sb : testSubs) {
        const u32 m = sb.second - sb.first;
        const DescView h(dv.h_desc, m);
        size_t o = 0;
        for (u32 q = 0; q < m; q++) {
          const u32 i = sb.first + q;
          h.srcOff[q] = off[i] - off[sb.first]; h.srcSize[q] = sizes[i]; h.dstCap[q] = (u32)encode_bound(sizes[i]); h.dstOff[q] = o; o += align_up(h.dstCap[q], 16);
        }
        DTCK(cudaMemcpyAsync(dv.d_desc, dv.h_desc, DescView::bytes(m), cudaMemcpyHostToDevice, st));
        const Items it = DescView(dv.d_desc, m).items(dSamples + off[sb.first], dv.d_dst, dv.d_result);
        int nl = 0;
        DTCK(encode_launch(encode_args(it, m, 0, level, 0, testMax, ENC_EXCLUSIVE, dEnc, &enc), *dv.enc, st, &nl));
        dv.launches += nl;
        DTCK(cudaMemcpyAsync(dv.h_result, dv.d_result, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
        DTCK(cudaStreamSynchronize(st));
        for (u32 q = 0; q < m; q++) score += is_err(dv.h_result[q]) ? sizes[sb.first + q] : dv.h_result[q];
      }
    }
    if (score < bestScore) { bestScore = score; bestK = sa.k[c]; best.assign(out.begin(), out.begin() + size); }
  }
  memcpy(dict, best.data(), best.size());
  pr.k = bestK; pr.d = d;
  return (u32)best.size();
}

}  // namespace zb
