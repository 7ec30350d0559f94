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
