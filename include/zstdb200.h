/* zstdb200.h — C ABI of libzstdb200, the B200-native batched Zstandard frame codec.
 *
 * This is the drop-in boundary for the hot path of epam/Zstandard (reference at /root/reference): the managed
 * host keeps its public API and binds these entry points through P/Invoke (C#) or JNI/Panama (Java); see
 * INTEGRATION.md for the stubs.  Every entry point names the reference interface it stands behind.
 *
 * Result convention — identical to the reference (csharp/src/ZStdErrors.cs:61-100): a per-item `uint32_t` is
 * either the number of bytes written or `(uint32_t)-(uint32_t)code`; it is an error iff it is greater than
 * (uint32_t)-120.  Codes: GENERIC 1, prefix_unknown 10, frameParameter_unsupported 14,
 * frameParameter_windowTooLarge 16, corruption_detected 20, checksum_wrong 22, dictionary_corrupted 30,
 * dictionary_wrong 32, dstSize_tooSmall 70, srcSize_wrong 72.
 * The `int` returned by batch calls is for batch-level failures only (0 = ok; CUDA error, bad argument, arena
 * too small): one bad item never fails the batch.
 *
 * There is no CPU fallback: every call that decodes or encodes runs CUDA kernels on the devices of the context
 * and fails if none is usable.
 */
#ifndef ZSTDB200_H
#define ZSTDB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct zstdb200_ctx zstdb200_ctx;

/* Creates a context owning, per listed device: one CUDA stream set, device staging for `max_batch_bytes` of
 * uncompressed data per in-flight sub-batch, the decoder's scratch arenas and pinned host staging.
 * devices == NULL or n_devices == 0 selects device 0.  Larger batches are processed in several sub-batches.
 * A context is single-caller; several contexts may be used concurrently.
 * (No reference counterpart: the reference allocates a ZSTD_DCtx per call, ZStdDecompress.cs:2174-2180.) */
int zstdb200_create(zstdb200_ctx** out, const int* devices, int n_devices, size_t max_batch_bytes);
void zstdb200_destroy(zstdb200_ctx* ctx);
/* Text of the last batch-level failure on this context ("" if none). */
const char* zstdb200_last_error(const zstdb200_ctx* ctx);

/* ZStdDecompress.GetDecompressedSize(byte[] src, uint srcSize) — csharp/src/ZStdDecompress.cs:590-622
 * (Java: ZstdDecompressor.getDecompressedSize, java/.../ZstdDecompressor.java:30-33).  Host-only header parse.
 * Returns 0 when the size is unknown, the header is invalid/incomplete or the frame is skippable. */
uint64_t zstdb200_get_decompressed_size(const void* src, uint32_t srcSize);

/* ZStdErrors.IsError — csharp/src/ZStdErrors.cs:97-100 (internal in the reference; exported for hosts). */
int zstdb200_is_error(uint32_t code);

/* ZStdDecompress.Decompress(byte[] dst, uint dstCapacity, byte[] src, uint srcSize) —
 * csharp/src/ZStdDecompress.cs:2182-2186 (Java: ZstdDecompressor.decompress, ZstdDecompressor.java:22-28).
 * One item through the batched path (n = 1): one descriptor copy, the kernels, the output copy, one synchronisation.
 * A NULL dst or src is an empty array (capacity / size taken as 0).  Returns the reference's result code. */
uint32_t zstdb200_decompress(zstdb200_ctx* ctx, void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize);

/* ZSTD_decompress_usingDict — csharp/src/ZStdDecompress.cs:2162-2167, dictionary loading :2366-2475 (present in the
 * reference but unreachable from its public API, which passes no dictionary, :2171; SURVEY.md §8f-3).  The dictionary
 * becomes part of the context: every later zstdb200_decompress* call starts each data frame from it (content as the
 * window's prefix; for a dictionary with magic 0xEC30A437 also its Huffman table, sequence tables and repeat offsets).
 * A malformed entropy section makes every data frame fail with dictionary_corrupted; a frame that names another
 * dictionary id fails with dictionary_wrong — the reference's codes.  dict == NULL or dictSize == 0 removes it.
 * The bytes are copied; returns 0, or non-zero on a CUDA / allocation failure (zstdb200_last_error). */
int zstdb200_load_dictionary(zstdb200_ctx* ctx, const void* dict, uint32_t dictSize);

/* Batched overload of the same call: item i decodes src[i][0..srcSize[i]) into dst[i][0..dstCap[i]) and stores
 * its result code in result[i].  Host pointers; the call returns after all outputs are in host memory.
 * Items are sharded over the context's devices by bytes; there is no cross-device traffic.
 * dstCap[i] may exceed max_batch_bytes (a large reusable scratch buffer): the device-side capacity is what the item
 * can produce; only an item whose CONTENT exceeds the context's arenas fails the call.
 * Bytes of dst[i] past result[i] are unspecified after the call when dst buffers lie back to back in pinned memory
 * (they are DMA'd as one span); on an error result the output is unspecified (the reference leaves a partial decode). */
int zstdb200_decompress_batch(zstdb200_ctx* ctx, const void* const* src, const uint32_t* srcSize,
                              void* const* dst, const uint32_t* dstCap, uint32_t* result, size_t n);

/* Device-resident variant for pipelines that already hold frames in HBM (and for roofline measurement).
 * All pointers are device pointers on device `devices[device_index]`; item i is
 * src_base[src_off[i] .. +src_size[i]) -> dst_base[dst_off[i] .. +dst_cap[i]).  Requirements: dst_off is
 * non-decreasing with dst_off[i] + dst_cap[i] <= dst_off[i+1]; dst_off[n-1] + dst_cap[n-1] <= max_batch_bytes;
 * n <= zstdb200_max_items(ctx).  Work is enqueued on `stream` (a cudaStream_t, NULL = the context's stream).
 * Items that hold several data frames (DecompressMultiFrame, ZStdDecompress.cs:2096-2160) take one pass of the
 * kernels per data frame; the count of such items has to reach the host, so this call synchronises `stream`
 * once per pass (once in total when every item holds a single data frame) before it returns. */
int zstdb200_decompress_batch_device(zstdb200_ctx* ctx, int device_index,
                                     const void* src_base, const uint64_t* src_off, const uint32_t* src_size,
                                     void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                     uint32_t* result, size_t n, void* stream);

/* Compression (no reference counterpart exists: epam/Zstandard ships no compressor, SURVEY.md §0 F1; the
 * signatures mirror the decompress side).  level 1..3, or -7..-1: libzstd's fast negative levels
 * (ZSTD_c_compressionLevel = -N, zstd --fast=N), faster and larger, with literals stored raw; any other level is a batch-level
 * failure.  checksum != 0 appends the XXH64 content checksum.  Frames are standard zstd frames accepted by the reference
 * decoder. */
size_t zstdb200_compress_bound(size_t srcSize);
uint32_t zstdb200_compress(zstdb200_ctx* ctx, int level, int checksum, void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize);
int zstdb200_compress_batch(zstdb200_ctx* ctx, int level, int checksum,
                            const void* const* src, const uint32_t* srcSize,
                            void* const* dst, const uint32_t* dstCap, uint32_t* result, size_t n);
/* Device-pointer variant.  Requirements (the encoder's scratch arenas are addressed from src_off, nothing is
 * validated on the device): src_off is non-decreasing with src_off[i] + src_size[i] <= src_off[i+1];
 * src_off[n-1] + src_size[n-1] <= max_batch_bytes; the source is readable 8 bytes past its last item; dst ranges do
 * not overlap; n <= zstdb200_max_items(ctx).  The call fetches src_size once (one small copy, one synchronisation of
 * `stream`) to size the match finder's tables by the largest chunk, then only enqueues. */
int zstdb200_compress_batch_device(zstdb200_ctx* ctx, int device_index, int level, int checksum,
                                   const void* src_base, const uint64_t* src_off, const uint32_t* src_size,
                                   void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                   uint32_t* result, size_t n, void* stream);

/* The same three calls with the context's dictionary (the one zstdb200_load_dictionary loaded; same arguments, levels 1..3 and
 * -7..-1, and contracts as the call each mirrors).  Frames name the dictionary's id in their header (a raw-content dictionary has id 0 and none is
 * written), match against its content and start from its repeat offsets; they decode with that dictionary
 * (zstdb200_decompress*, libzstd's ZSTD_decompress_usingDict).  With no dictionary loaded the call fails at batch level
 * (non-zero, or GENERIC for zstdb200_compress_using_dict; zstdb200_last_error says why); when the dictionary's entropy
 * section is malformed every item gets dictionary_corrupted.  The calls without _using_dict ignore a loaded dictionary. */
uint32_t zstdb200_compress_using_dict(zstdb200_ctx* ctx, int level, int checksum, void* dst, uint32_t dstCapacity, const void* src, uint32_t srcSize);
int zstdb200_compress_batch_using_dict(zstdb200_ctx* ctx, int level, int checksum,
                                       const void* const* src, const uint32_t* srcSize,
                                       void* const* dst, const uint32_t* dstCap, uint32_t* result, size_t n);
int zstdb200_compress_batch_device_using_dict(zstdb200_ctx* ctx, int device_index, int level, int checksum,
                                              const void* src_base, const uint64_t* src_off, const uint32_t* src_size,
                                              void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                              uint32_t* result, size_t n, void* stream);

/* Dictionary training (no reference counterpart: users of the reference train with libzstd's ZDICT_trainFromBuffer).  Builds
 * a dictionary with entropy tables (magic 0xEC30A437) from nbSamples samples laid back to back in host memory, as ZDICT takes
 * them.  The content is selected as libzstd 1.5.5's fastCover trainer selects it (ZDICT_trainFromBuffer_fastCover with a
 * fixed k; with k = 0 the k search of ZDICT_trainFromBuffer, candidates scored by compressing the test share of the samples
 * with this library's dictionary encoder at `level`); the entropy tables come from this library's match stage over the first
 * block of the finalize samples.  Runs on the context's first device, allocates what the sample set needs and frees it before
 * returning; the context's loaded dictionary is not touched.  Returns the dictionary size or an error code:
 * dstSize_tooSmall (capacity below 256 or below k; 1998 when searching), srcSize_wrong (fewer than 5 training samples, no
 * test sample when searching, fewer bytes than max(d, 8)), GENERIC with zstdb200_last_error set (a parameter out of range,
 * samples totalling 2^32 bytes or more, a test sample larger than max_batch_bytes, a CUDA failure). */
typedef struct {
  uint32_t k;             /* segment size; 0 = search k over ZDICT_trainFromBuffer's grid {50, 537, 1024, 1511, 1998}; at most 2048 */
  uint32_t d;             /* d-mer size, 6 or 8; 0 = 8 */
  uint32_t f;             /* log2 of the frequency table; 0 = 20; at most 24 */
  uint32_t accel;         /* 1..10, ZDICT's fastCover acceleration; 0 = 1 */
  uint32_t split_percent; /* training share of the samples; 0 = 75 when searching, 100 with a fixed k (ZDICT's defaults) */
  int      level;         /* 1..3: level whose match stage gathers the entropy statistics and scores search candidates; 0 = 3 */
  uint32_t dict_id;       /* 0 = ZDICT's rule (XXH64 of the selected content, mod 2^31 - 32768, + 32768) */
} zstdb200_train_params;

uint32_t zstdb200_train_dictionary(zstdb200_ctx* ctx, void* dictBuffer, uint32_t dictCapacity,
                                   const void* samples, const uint32_t* sampleSizes, size_t nbSamples,
                                   zstdb200_train_params* params /* NULL = defaults; k and d chosen are written back */);

/* Seekable archives (no reference counterpart; zstd's seekable format, contrib/seekable_format/
 * zstd_seekable_compression_format.md in the zstd repository).  An archive is independent zstd frames back to back from
 * byte 0, followed by a skippable frame (magic 0x184D2A5E) holding the seek table: per frame its Compressed_Size,
 * Decompressed_Size and, when the descriptor's bit 7 is set, the low 32 bits of the XXH64 of its content; then
 * Number_Of_Frames, the descriptor byte and 0x8F92EAB1.  Any zstd decoder reads such an archive (concatenated frames, the
 * table skipped), zstdb200_decompress included; the calls below decode any byte range of it with the frames that cover the
 * range as items of one batch. */
typedef struct {
  uint64_t content_size;        /* sum of Decompressed_Size */
  uint64_t data_size;           /* bytes of the data frames (the archive without its seek table) */
  uint32_t n_frames;
  uint32_t checksums;           /* checksum flag of the descriptor */
  uint32_t max_frame_content, max_frame_compressed;
} zstdb200_seekable_info;

/* Host-only: reads the footer and the table of the archive src[0..srcSize).  Returns 0, or an error code (nothing else is
 * written): srcSize_wrong (shorter than 17 bytes; the table is longer than the archive), prefix_unknown (footer magic;
 * skippable magic), corruption_detected (a reserved descriptor bit 6..2 set; Frame_Size does not match the frame count and
 * entry size; the Compressed_Size values do not add up to exactly the bytes before the table).  Bits 1..0 are ignored. */
uint32_t zstdb200_seekable_info_get(const void* src, uint64_t srcSize, zstdb200_seekable_info* info);

/* Largest archive zstdb200_compress_seekable* writes for srcSize bytes in frames of frameSize (0 for frameSize 0). */
uint64_t zstdb200_seekable_bound(uint64_t srcSize, uint32_t frameSize);

/* Compresses src[0..srcSize) into one archive at dst and stores its size in *dstSize.  Frame i holds bytes
 * [i * frameSize, min((i + 1) * frameSize, srcSize)) and is byte for byte what zstdb200_compress_batch writes for that chunk
 * at the same level (1..3, -7..-1) and checksum.  checksum != 0: every frame carries its content checksum and the table the
 * same 4 bytes, with the checksum flag set; checksum == 0: neither does.  srcSize == 0 gives the 17-byte table frame alone.
 * Batch-level failures (non-zero, zstdb200_last_error), detected before any work starts: 1 <= frameSize <= max_batch_bytes
 * does not hold, more frames than the table's 32-bit Frame_Size holds (357 913 940 with checksums, 536 870 910 without),
 * dstCapacity < zstdb200_seekable_bound(srcSize, frameSize), a null pointer, a bad level.
 * Host variant: any srcSize within that frame count, over the sub-batches and devices of zstdb200_compress_batch; each
 * sub-batch's frames are packed on the device and cross PCIe once, back to back, into their final place (no per-frame
 * spare capacity, no second pass over the output). */
int zstdb200_compress_seekable(zstdb200_ctx* ctx, int level, int checksum, uint32_t frameSize,
                               const void* src, uint64_t srcSize, void* dst, uint64_t dstCapacity, uint64_t* dstSize);
/* Device variant: src, dst and dstSize are device pointers on device `devices[device_index]`.  Requires srcSize <=
 * max_batch_bytes and a frame count <= zstdb200_max_items(ctx); the source is readable 8 bytes past its end.  The frames are
 * encoded into the context's device staging, then packed with their table into dst (*dstSize is written on the device;
 * 0 if a frame failed, which a capacity at the bound rules out).  The descriptors' upload synchronises `stream` once (as
 * zstdb200_compress_batch_device does); everything else is enqueued on `stream` (NULL = the context's stream). */
int zstdb200_compress_seekable_device(zstdb200_ctx* ctx, int device_index, int level, int checksum, uint32_t frameSize,
                                      const void* src, uint64_t srcSize, void* dst, uint64_t dstCapacity,
                                      uint64_t* dstSize, void* stream);

/* Decodes content bytes [offset, offset + length) of the archive src[0..srcSize) into dst[0..length); no byte of dst outside
 * that range is written.  Only the frames that overlap the range are decoded, all as items of one batch (one launch
 * sequence of the decode pipeline per arena-sized round, never one pass per frame).  Frames inside the range decode straight
 * into dst; the first and last, when only part of them is in the range, decode into scratch and their in-range part is
 * copied out.  *code: 0, or the first error in archive order — a table error (the codes of zstdb200_seekable_info_get);
 * srcSize_wrong when the range ends past content_size (nothing is decoded); a frame's own decoder code; corruption_detected
 * when a frame decodes to a size other than its Decompressed_Size; checksum_wrong when the table's checksum does not match
 * (compared with the frame's own verified checksum when it has one, else with the XXH64 of its decoded bytes).  On an
 * error code the range's bytes are unspecified.  Batch-level failure (non-zero): a selected frame larger than
 * max_batch_bytes, a null pointer, a CUDA failure.  Host variant: host pointers; the plan runs through the host batch path
 * (items are spans of the archive, checked on the device right after their decode). */
int zstdb200_decompress_seekable(zstdb200_ctx* ctx, void* dst, uint64_t offset, uint64_t length,
                                 const void* src, uint64_t srcSize, uint32_t* code);
/* Device variant: dst, src and code are device pointers.  The footer and then the table are copied to the host (two small
 * copies, two synchronisations of `stream`); after that the call only enqueues (a range whose frames exceed one descriptor
 * upload of max_items frames waits for the previous upload's work once per further upload).  The queued work uses the
 * context's staging and scratch on that device, so the next call on the context that needs them first waits for it; a
 * caller never has to synchronise `stream` before making another call. */
int zstdb200_decompress_seekable_device(zstdb200_ctx* ctx, int device_index, void* dst, uint64_t offset, uint64_t length,
                                        const void* src, uint64_t srcSize, uint32_t* code, void* stream);

/* Pinned host memory for src/dst buffers (lets the batch calls DMA straight from/to caller memory). */
void* zstdb200_host_alloc(size_t bytes);
void zstdb200_host_free(void* p);

/* Introspection used by the bench harness. */
size_t zstdb200_max_items(const zstdb200_ctx* ctx);
int zstdb200_device_count(const zstdb200_ctx* ctx);
uint64_t zstdb200_kernel_launches(const zstdb200_ctx* ctx);   /* kernels launched by this context so far */
const char* zstdb200_version(void);
/* zstdb200_decompress_batch_device with CUDA events between its kernels; synchronises and returns the device
 * time of each kernel in kernel_ms[0..min(max_kernels, count)) (names via zstdb200_decode_kernel_name). */
int zstdb200_decompress_batch_device_timed(zstdb200_ctx* ctx, int device_index,
                                           const void* src_base, const uint64_t* src_off, const uint32_t* src_size,
                                           void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                           uint32_t* result, size_t n, void* stream, float* kernel_ms, int max_kernels);
const char* zstdb200_decode_kernel_name(int k);
int zstdb200_compress_batch_device_timed(zstdb200_ctx* ctx, int device_index, int level, int checksum,
                                         const void* src_base, const uint64_t* src_off, const uint32_t* src_size,
                                         void* dst_base, const uint64_t* dst_off, const uint32_t* dst_cap,
                                         uint32_t* result, size_t n, void* stream, float* kernel_ms, int max_kernels);
const char* zstdb200_encode_kernel_name(int k);

#ifdef __cplusplus
}
#endif
#endif /* ZSTDB200_H */
