// tests/hostsim/dict_train.cpp — CPU emulation of dictionary training (zstdb200_train_dictionary) (TEST AID ONLY).
//
// The serial statement of what the training kernels compute: the fastCover frequency pass and segment selection written
// straight from libzstd's loop (the reference the parallel scoring of k_dt_select is held to), the match stage over the first
// block of each finalize sample (dict_encoder.cpp's lock-step emulation of k_enc_match<DFAST, true>), its symbol histograms,
// and the shared table writer of zb_dict_train.cuh.  The k search scores each candidate by compressing the test samples with
// dict_encoder.cpp's emulation of the dictionary encoder.  tests/test_dictionary_train.py builds this file into its own library
// and compares it with ZDICT (selection, id, validity, ratio) and, on a GPU, with the library byte for byte.
#include "dict_encoder.cpp"
#include "../../zstandard_b200/csrc/zb_dict_train.cuh"

namespace {

struct TrainIn {
  const u8* samples; const u32* sizes; u32 n;
  std::vector<u64> off;   // off[i] = start of sample i, off[n] = total
  u32 nbTrain, nbTest;    // nbTest = 0 without a split
};

// FASTCOVER_computeFrequency over the training samples
void frequencies(const TrainIn& in, u32 f, u32 d, u32 skip, std::vector<u32>& freqs) {
  freqs.assign((size_t)1 << f, 0);
  const u32 readLen = d > 8 ? d : 8;
  for (u32 i = 0; i < in.nbTrain; i++)
    for (u64 p = in.off[i]; p + readLen <= in.off[i + 1]; p += skip + 1) freqs[dt_hash(in.samples + p, f, d)]++;
}

// The selection loop (FASTCOVER_buildDictionary / FASTCOVER_selectSegment): epochs round robin, the best window of each, its
// frequencies zeroed, its bytes copied to the tail of the buffer.  (Unlike COVER, fastCover does not trim zero-frequency
// d-mers off the window's ends.)  Returns the tail (the selection is buf[tail, capacity)).
u32 select_serial(const TrainIn& in, std::vector<u32>& freqs, u32 f, u32 k, u32 d, u32 capacity, std::vector<u8>& buf) {
  buf.assign(capacity, 0);
  const u32 readLen = d > 8 ? d : 8;
  const u64 trainBytes = in.off[in.nbTrain];
  const u32 nbDmers = (u32)(trainBytes - readLen + 1);
  const DtEpochs ep = dt_epochs(capacity, nbDmers, k);
  const u32 L = k - d + 1;
  std::vector<u16> segFreq((size_t)1 << f, 0);
  u32 tail = capacity, zeroRun = 0;
  for (u32 epoch = 0; tail > 0 && ep.num; epoch = (epoch + 1) % ep.num) {
    const u32 b = epoch * ep.size, e = b + ep.size;
    // slide the window [begin, end) over the epoch; the best one is the first that reaches the highest score
    u32 begin = b, end = b; u64 score = 0, best = 0; u32 bestB = 0, bestE = 0;
    while (end < e) {
      const u32 h = dt_hash(in.samples + end, f, d);
      if (segFreq[h] == 0) score += freqs[h];
      end++; segFreq[h]++;
      if (end - begin == L + 1) {
        const u32 hd = dt_hash(in.samples + begin, f, d);
        if (--segFreq[hd] == 0) score -= freqs[hd];
        begin++;
      }
      if (score > best) { best = score; bestB = begin; bestE = end; }
    }
    for (; begin < end; begin++) segFreq[dt_hash(in.samples + begin, f, d)]--;
    if (best == 0) { if (++zeroRun >= DT_ZERO_SCORE_RUN) break; continue; }
    zeroRun = 0;
    for (u32 p = bestB; p < bestE; p++) freqs[dt_hash(in.samples + p, f, d)] = 0;
    const u32 len = std::min(bestE - bestB + d - 1, tail);
    if (len < d) break;
    tail -= len;
    memcpy(buf.data() + tail, in.samples + bestB, len);
  }
  return tail;
}

// Match stage over the first block of each finalize sample against the raw-content dictionary of the selection, and the
// histograms of what it produced
void gather_stats(const TrainIn& in, const u8* sel, u32 selSize, u32 nFinal, int level, DtStats& st) {
  memset(&st, 0, sizeof st);
  DictState ds; dt_raw_dict_state(ds, selSize);
  std::vector<u8> selPad(sel, sel + selSize); selPad.resize((size_t)selSize + 64, 0);
  std::vector<u8> enc(enc_dict_bytes(selSize));
  static HufBuildWk wk; static HufFseScratch fs; static u8 slot[260], tableSymbol[512];
  enc_dict_prepare(selPad.data(), selSize, ds, reinterpret_cast<EncDict*>(enc.data()), wk, fs, slot, tableSymbol);
  const EncDict* ed = reinterpret_cast<const EncDict*>(enc.data());
  for (u32 i = 0; i < nFinal; i++) {
    const u32 size = std::min<u32>(in.sizes[i], BLOCKSIZE_MAX);
    std::vector<u8> padded((size_t)size + 64, 0);
    u8* src = padded.data() + 16;
    if (size) memcpy(src, in.samples + in.off[i], size);
    DictWarpMatcher m; m.src = src; m.size = size; m.dfast = level >= 3; m.hlogL = enc_hlog_long(level, false);
    m.hlogS = enc_hlog_short(level, false); m.mls = level <= 1 ? 6 : 5;
    m.tab.assign((1u << m.hlogL) + (1u << m.hlogS), 0);
    m.ed = ed; m.rep1 = ed->rep[0]; m.rep2 = ed->rep[1];
    bool rle = size >= 2;
    for (u32 q = 1; q < size && rle; q++) if (src[q] != src[0]) rle = false;
    SeqStore s; s.n = 0; s.nlits = 0;
    if (!m(s, 0, src, size, rle)) continue;
    for (u32 q = 0; q < s.nlits; q++) st.lit[s.lits[q]]++;
    for (u32 q = 0; q < s.n; q++) {
      u32 ll, ob, mlm3; seq_get(s, q, ll, ob, mlm3);
      st.ll[ll_code(ll)]++; st.ml[ml_code(mlm3)]++; st.of[highbit(ob)]++;
    }
  }
}

// Selection -> finished dictionary in out (capacity bytes); returns its size
u32 finalize(const TrainIn& in, const u8* sel, u32 selSize, u32 capacity, u32 accel, int level, u32 dictID, u8* out) {
  DtStats st;
  gather_stats(in, sel, selSize, (u32)((u64)in.nbTrain * dt_accel_finalize(accel) / 100), level, st);
  static DtHeaderScratch w;
  u8 hdr[DT_DICT_MIN];
  const u32 h = dt_write_header(hdr, dictID ? dictID : dt_dict_id(sel, selSize), st, selSize, w);
  if (!h) return zerr(ZE_GENERIC);
  return dt_assemble(out, capacity, hdr, h, sel, selSize);
}

// Sum of the frame sizes of the test samples compressed with the dictionary (as zstdb200_compress_batch_using_dict; batch_max:
// the largest test sample)
u64 score_dictionary(const TrainIn& in, const u8* dict, u32 size, int level) {
  std::vector<u8> bytes(dict, dict + size); bytes.resize((size_t)size + 64, 0);
  DictState ds; static HufBuildWk wk; static HufFseScratch fs; static u8 slot[260], tableSymbol[512]; static s16 norm[64]; static u16 next[64];
  dict_load(bytes.data(), size, ds, wk, fs, slot, norm, next);
  std::vector<u8> enc(enc_dict_bytes(ds.err ? 0 : ds.contentSize));
  enc_dict_prepare(bytes.data(), size, ds, reinterpret_cast<EncDict*>(enc.data()), wk, fs, slot, tableSymbol);
  u32 batchMax = 0;
  for (u32 i = in.nbTrain; i < in.n; i++) batchMax = std::max(batchMax, in.sizes[i]);
  u64 total = 0;
  std::vector<u8> dst;
  for (u32 i = in.nbTrain; i < in.n; i++) {
    dst.resize((size_t)in.sizes[i] + (in.sizes[i] >> 8) + 32 + 3 * ((in.sizes[i] >> 17) + 1));   // encode_bound
    const u32 r = compress(dst.data(), (u32)dst.size(), in.samples + in.off[i], in.sizes[i], level, 0, batchMax, reinterpret_cast<const EncDict*>(enc.data()));
    total += is_err(r) ? in.sizes[i] : r;
  }
  return total;
}

}  // namespace

// Selection only, for a fixed k (split_percent 0 = 100): the content section ZDICT builds before it finalizes.  Returns its size
// (written to the end of sel[0..capacity)) or an error code.
extern "C" uint32_t dtsim_select(uint8_t* sel, uint32_t capacity, const uint8_t* samples, const uint32_t* sizes, uint32_t n,
                                 uint32_t k, uint32_t d, uint32_t f, uint32_t accel, uint32_t split_percent) {
  TrainIn in; in.samples = samples; in.sizes = sizes; in.n = n; in.off.assign(n + 1, 0);
  for (u32 i = 0; i < n; i++) in.off[i + 1] = in.off[i] + sizes[i];
  if (!split_percent) split_percent = 100;
  in.nbTrain = split_percent < 100 ? (u32)((double)n * ((double)split_percent / 100.0)) : n;
  if (in.nbTrain < 5 || in.off[n] < 8) return zerr(ZE_srcSize_wrong);
  std::vector<u32> freqs; std::vector<u8> buf;
  frequencies(in, f, d, dt_accel_skip(accel), freqs);
  const u32 tail = select_serial(in, freqs, f, k, d, capacity, buf);
  memcpy(sel + tail, buf.data() + tail, capacity - tail);
  return capacity - tail;
}

// The whole of zstdb200_train_dictionary on the CPU, parameters as in include/zstdb200.h (already validated by the caller:
// the Python test passes what the library accepts).  params[0..7) = k, d, f, accel, split_percent, level, dict_id; k and d
// chosen are written back.  Returns the dictionary size or an error code.
extern "C" uint32_t dtsim_train(uint8_t* dict, uint32_t capacity, const uint8_t* samples, const uint32_t* sizes, uint32_t n,
                                uint32_t* params) {
  const u32 k0 = params[0], d = params[1] ? params[1] : 8, f = params[2] ? params[2] : 20, accel = params[3] ? params[3] : 1;
  const u32 split = params[4] ? params[4] : (k0 ? 100 : 75);
  const int level = params[5] ? (int)params[5] : 3;
  const u32 dictID = params[6];
  TrainIn in; in.samples = samples; in.sizes = sizes; in.n = n; in.off.assign(n + 1, 0);
  for (u32 i = 0; i < n; i++) in.off[i + 1] = in.off[i] + sizes[i];
  in.nbTrain = split < 100 ? (u32)((double)n * ((double)split / 100.0)) : n;
  in.nbTest = split < 100 ? n - in.nbTrain : 0;
  if (capacity < DT_DICT_MIN || capacity < (k0 ? k0 : dt_search_k(DT_SEARCH_KS - 1))) return zerr(ZE_dstSize_tooSmall);
  if (in.off[n] < (d > 8 ? d : 8) || in.nbTrain < 5 || (!k0 && in.nbTest < 1)) return zerr(ZE_srcSize_wrong);
  if (in.off[in.nbTrain] < (d > 8 ? d : 8)) return zerr(ZE_srcSize_wrong);
  std::vector<u32> freqs0, freqs; std::vector<u8> buf, out(capacity), best;
  frequencies(in, f, d, dt_accel_skip(accel), freqs0);
  u64 bestScore = ~0ull; u32 bestK = 0;
  for (u32 c = 0; c < (k0 ? 1u : DT_SEARCH_KS); c++) {
    const u32 k = k0 ? k0 : dt_search_k(c);
    freqs = freqs0;
    const u32 tail = select_serial(in, freqs, f, k, d, capacity, buf);
    const u32 size = finalize(in, buf.data() + tail, capacity - tail, capacity, accel, level, dictID, out.data());
    if (is_err(size)) return size;
    const u64 score = k0 ? 0 : score_dictionary(in, out.data(), size, level);
    if (score < bestScore) { bestScore = score; bestK = k; best.assign(out.begin(), out.begin() + size); }
  }
  memcpy(dict, best.data(), best.size());
  params[0] = bestK; params[1] = d;
  return (u32)best.size();
}
