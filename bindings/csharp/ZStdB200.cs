// ZStdB200.cs - the reference's public C# surface (csharp/src/ZStdDecompress.cs:590-607, 2182-2191) over libzstdb200.
//
// Drop-in for the bodies of EPAM.Deltix.ZStd.ZStdDecompress: same method names, argument meaning and result convention
// (bytes written, or (uint)-code with the codes of ZStdErrors.cs:61-100).  New next to them: batched overloads, a
// dictionary entry point (the reference keeps ZSTD_decompress_usingDict internal, :2162-2171) and ZStdCompress (the
// reference ships no compressor).  Target framework netstandard2.0 like the reference (Zstandard.csproj:3): no Span,
// no newer allocation APIs.  There is no CPU fallback: without a CUDA device the first call throws.
using System;
using System.Collections.Generic;
using System.Runtime.InteropServices;

namespace EPAM.Deltix.ZStd
{
    internal static unsafe class Native
    {
        const string Lib = "zstdb200";   // libzstdb200.so
        [DllImport(Lib)] internal static extern int zstdb200_create(out IntPtr ctx, int* devices, int nDevices, UIntPtr maxBatchBytes);
        [DllImport(Lib)] internal static extern void zstdb200_destroy(IntPtr ctx);
        [DllImport(Lib)] internal static extern IntPtr zstdb200_last_error(IntPtr ctx);
        [DllImport(Lib)] internal static extern ulong zstdb200_get_decompressed_size(void* src, uint srcSize);
        [DllImport(Lib)] internal static extern int zstdb200_is_error(uint code);
        [DllImport(Lib)] internal static extern uint zstdb200_decompress(IntPtr ctx, void* dst, uint dstCapacity, void* src, uint srcSize);
        [DllImport(Lib)] internal static extern int zstdb200_load_dictionary(IntPtr ctx, void* dict, uint dictSize);
        [DllImport(Lib)] internal static extern int zstdb200_decompress_batch(IntPtr ctx, void** src, uint* srcSize, void** dst, uint* dstCap, uint* result, UIntPtr n);
        [DllImport(Lib)] internal static extern UIntPtr zstdb200_compress_bound(UIntPtr srcSize);
        [DllImport(Lib)] internal static extern uint zstdb200_compress(IntPtr ctx, int level, int checksum, void* dst, uint dstCapacity, void* src, uint srcSize);
        [DllImport(Lib)] internal static extern int zstdb200_compress_batch(IntPtr ctx, int level, int checksum, void** src, uint* srcSize, void** dst, uint* dstCap, uint* result, UIntPtr n);
        [DllImport(Lib)] internal static extern uint zstdb200_compress_using_dict(IntPtr ctx, int level, int checksum, void* dst, uint dstCapacity, void* src, uint srcSize);
        [DllImport(Lib)] internal static extern int zstdb200_compress_batch_using_dict(IntPtr ctx, int level, int checksum, void** src, uint* srcSize, void** dst, uint* dstCap, uint* result, UIntPtr n);
        [DllImport(Lib)] internal static extern IntPtr zstdb200_host_alloc(UIntPtr bytes);
        [DllImport(Lib)] internal static extern void zstdb200_host_free(IntPtr p);
        [DllImport(Lib)] internal static extern IntPtr zstdb200_version();
        [DllImport(Lib)] internal static extern uint zstdb200_train_dictionary(IntPtr ctx, void* dictBuffer, uint dictCapacity, void* samples, uint* sampleSizes, UIntPtr nbSamples, TrainParams* parameters);

        // one context per thread: a zstdb200_ctx is single-caller (include/zstdb200.h)
        [ThreadStatic] static IntPtr ctx;
        internal static IntPtr Ctx()
        {
            if (ctx == IntPtr.Zero && zstdb200_create(out ctx, null, 0, (UIntPtr)(256u << 20)) != 0)
                throw new InvalidOperationException("libzstdb200: no usable CUDA device (there is no CPU fallback)");
            return ctx;
        }
        internal static void Check(int rc)
        {
            if (rc != 0) throw new InvalidOperationException(Marshal.PtrToStringAnsi(zstdb200_last_error(Ctx())));
        }

        internal delegate int BatchCall(void** src, uint* srcSize, void** dst, uint* dstCap, uint* result, UIntPtr n);

        // pins every segment, builds the descriptor tables in native memory (n may be tens of thousands: no stackalloc)
        internal static void Batch(IReadOnlyList<ArraySegment<byte>> srcs, IReadOnlyList<ArraySegment<byte>> dsts, uint[] results, BatchCall call)
        {
            int n = srcs.Count;
            if (dsts.Count != n || results.Length < n) throw new ArgumentException("srcs, dsts and results must have one entry per item");
            var pins = new GCHandle[2 * n];
            IntPtr tables = Marshal.AllocHGlobal((IntPtr)((long)Math.Max(n, 1) * (2 * sizeof(void*) + 2 * sizeof(uint))));
            void** sp = (void**)tables; void** dp = sp + n; uint* ss = (uint*)(dp + n); uint* dc = ss + n;
            try
            {
                for (int i = 0; i < n; i++)
                {
                    // a null or empty array is an empty item (the library takes NULL with size 0)
                    if (srcs[i].Array != null && srcs[i].Count > 0)
                    {
                        pins[2 * i] = GCHandle.Alloc(srcs[i].Array, GCHandleType.Pinned);
                        sp[i] = (byte*)pins[2 * i].AddrOfPinnedObject() + srcs[i].Offset;
                    }
                    else sp[i] = null;
                    if (dsts[i].Array != null && dsts[i].Count > 0)
                    {
                        pins[2 * i + 1] = GCHandle.Alloc(dsts[i].Array, GCHandleType.Pinned);
                        dp[i] = (byte*)pins[2 * i + 1].AddrOfPinnedObject() + dsts[i].Offset;
                    }
                    else dp[i] = null;
                    ss[i] = srcs[i].Array == null ? 0u : (uint)srcs[i].Count;
                    dc[i] = dsts[i].Array == null ? 0u : (uint)dsts[i].Count;
                }
                fixed (uint* r = results) Check(call(sp, ss, dp, dc, r, (UIntPtr)n));
            }
            finally
            {
                foreach (var h in pins) if (h.IsAllocated) h.Free();
                Marshal.FreeHGlobal(tables);
            }
        }
    }

    public static unsafe class ZStdDecompress
    {
        // ZStdDecompress.cs:590-607 - unchanged signatures; a host-only header parse in the library
        public static ulong GetDecompressedSize(byte[] src) { return GetDecompressedSize(src, (uint)src.Length); }
        public static ulong GetDecompressedSize(byte[] src, uint srcSize)
        {
            fixed (byte* p = src) return Native.zstdb200_get_decompressed_size(p, srcSize);
        }

        // ZStdDecompress.cs:2182-2191 - unchanged signatures and result convention
        public static uint Decompress(byte[] dst, uint dstCapacity, byte[] src, uint srcSize)
        {
            if (dstCapacity > (uint)dst.Length || srcSize > (uint)src.Length) throw new ArgumentOutOfRangeException();
            fixed (byte* d = dst, s = src) return Native.zstdb200_decompress(Native.Ctx(), d, dstCapacity, s, srcSize);
        }
        public static uint Decompress(byte[] dst, byte[] src) { return Decompress(dst, (uint)dst.Length, src, (uint)src.Length); }

        public static bool IsError(uint code) { return Native.zstdb200_is_error(code) != 0; }   // ZStdErrors.cs:97-100

        // new: ZSTD_decompress_usingDict (ZStdDecompress.cs:2162-2167).  The dictionary stays with this thread's context
        // until replaced; null removes it.
        public static void UseDictionary(byte[] dict)
        {
            fixed (byte* p = dict) Native.Check(Native.zstdb200_load_dictionary(Native.Ctx(), p, dict == null ? 0u : (uint)dict.Length));
        }

        // new: batched overload - one independent item (one or more frames) per segment.  results[i] has the encoding of
        // the single-item call; an exception is a batch-level failure (CUDA error, bad argument).
        public static void Decompress(IReadOnlyList<ArraySegment<byte>> srcs, IReadOnlyList<ArraySegment<byte>> dsts, uint[] results)
        {
            IntPtr c = Native.Ctx();
            Native.Batch(srcs, dsts, results, (sp, ss, dp, dc, r, n) => Native.zstdb200_decompress_batch(c, sp, ss, dp, dc, r, n));
        }
    }

    // new class: the reference ships no compressor; same calling shape as the decoder
    public static unsafe class ZStdCompress
    {
        public static uint CompressBound(uint srcSize) { return (uint)Native.zstdb200_compress_bound((UIntPtr)srcSize); }

        public static uint Compress(byte[] dst, byte[] src, int level = 3, bool checksum = true)
        {
            fixed (byte* d = dst, s = src)
                return Native.zstdb200_compress(Native.Ctx(), level, checksum ? 1 : 0, d, (uint)dst.Length, s, (uint)src.Length);
        }

        // one frame per segment; levels 1-3 (fast / double-fast match finder) or -7..-1 (libzstd's fast negative levels: faster,
        // larger, literals stored raw), XXH64 content checksum on request
        public static void Compress(IReadOnlyList<ArraySegment<byte>> srcs, IReadOnlyList<ArraySegment<byte>> dsts, uint[] results, int level = 3, bool checksum = true)
        {
            IntPtr c = Native.Ctx();
            int cs = checksum ? 1 : 0;
            Native.Batch(srcs, dsts, results, (sp, ss, dp, dc, r, n) => Native.zstdb200_compress_batch(c, level, cs, sp, ss, dp, dc, r, n));
        }

        // with the dictionary of this thread's context (ZStdDecompress.UseDictionary): frames name its id and decode with it.
        // Without one the single-item call returns GENERIC and the batched call throws.
        public static uint CompressUsingDict(byte[] dst, byte[] src, int level = 3, bool checksum = true)
        {
            fixed (byte* d = dst, s = src)
                return Native.zstdb200_compress_using_dict(Native.Ctx(), level, checksum ? 1 : 0, d, (uint)dst.Length, s, (uint)src.Length);
        }
        public static void CompressUsingDict(IReadOnlyList<ArraySegment<byte>> srcs, IReadOnlyList<ArraySegment<byte>> dsts, uint[] results, int level = 3, bool checksum = true)
        {
            IntPtr c = Native.Ctx();
            int cs = checksum ? 1 : 0;
            Native.Batch(srcs, dsts, results, (sp, ss, dp, dc, r, n) => Native.zstdb200_compress_batch_using_dict(c, level, cs, sp, ss, dp, dc, r, n));
        }
    }

    // zstdb200_train_params (include/zstdb200.h); zero fields take the library's defaults
    [StructLayout(LayoutKind.Sequential)]
    public struct TrainParams
    {
        public uint K;             // 0 = search {50, 537, 1024, 1511, 1998}
        public uint D;             // 6 or 8; 0 = 8
        public uint F;             // 0 = 20; at most 24
        public uint Accel;         // 1..10; 0 = 1
        public uint SplitPercent;  // 0 = 75 when searching, 100 with a fixed k
        public int Level;          // 1..3; 0 = 3
        public uint DictId;        // 0 = derived from the content
    }

    public static unsafe class ZStdDictionary
    {
        // new: builds a dictionary (magic 0xEC30A437) from sample messages on this thread's context's GPU, as libzstd's fastCover
        // trainer selects content.  Returns its bytes; parameters (optional) receives the k and d chosen.  Throws on an error
        // result, with its code in the message.
        public static byte[] TrainDictionary(IReadOnlyList<ArraySegment<byte>> samples, int capacity, ref TrainParams parameters)
        {
            int n = samples.Count;
            long total = 0;
            for (int i = 0; i < n; i++) total += samples[i].Count;
            var blob = new byte[Math.Max(total, 1)];
            var sizes = new uint[Math.Max(n, 1)];
            long pos = 0;
            for (int i = 0; i < n; i++)
            {
                if (samples[i].Count > 0) Buffer.BlockCopy(samples[i].Array, samples[i].Offset, blob, (int)pos, samples[i].Count);
                sizes[i] = (uint)samples[i].Count; pos += samples[i].Count;
            }
            var dict = new byte[capacity];
            uint r;
            fixed (byte* d = dict, s = blob) fixed (uint* z = sizes) fixed (TrainParams* p = &parameters)
                r = Native.zstdb200_train_dictionary(Native.Ctx(), d, (uint)capacity, s, z, (UIntPtr)n, p);
            if (Native.zstdb200_is_error(r) != 0)
                throw new InvalidOperationException("zstdb200_train_dictionary failed: error " + (uint)(-(int)r) + " " + Marshal.PtrToStringAnsi(Native.zstdb200_last_error(Native.Ctx())));
            Array.Resize(ref dict, (int)r);
            return dict;
        }
        public static byte[] TrainDictionary(IReadOnlyList<ArraySegment<byte>> samples, int capacity)
        {
            var p = new TrainParams();
            return TrainDictionary(samples, capacity, ref p);
        }
    }

    // Pinned host memory for callers that assemble large batches themselves: buffers that lie back to back in one such
    // allocation take the library's direct-DMA path (INTEGRATION.md, "Behaviour notes for hosts").
    public sealed unsafe class PinnedBuffer : IDisposable
    {
        public IntPtr Pointer { get; private set; }
        public long Length { get; private set; }
        public PinnedBuffer(long bytes)
        {
            Pointer = Native.zstdb200_host_alloc((UIntPtr)(ulong)bytes);
            if (Pointer == IntPtr.Zero) throw new OutOfMemoryException("zstdb200_host_alloc");
            Length = bytes;
        }
        public void Dispose()
        {
            if (Pointer != IntPtr.Zero) { Native.zstdb200_host_free(Pointer); Pointer = IntPtr.Zero; }
            GC.SuppressFinalize(this);
        }
        ~PinnedBuffer() { if (Pointer != IntPtr.Zero) Native.zstdb200_host_free(Pointer); }
    }
}
