"""zstandard_b200 — host-side mirror of the epam/Zstandard public API over libzstdb200 (sm_100a CUDA).

The reference's host language is C# (`EPAM.Deltix.ZStd.ZStdDecompress`, csharp/src/ZStdDecompress.cs:37-42) and
no .NET toolchain exists in this image, so this package is the thin Python stand-in for the C# shim of
INTEGRATION.md: the same names, argument meaning and result convention, bound to the same C ABI
(include/zstdb200.h) through ctypes instead of P/Invoke.  All decoding/encoding happens in CUDA kernels inside
libzstdb200.so; there is no CPU path here — loading fails loudly when the library is missing and context
creation fails when no GPU is present.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libzstdb200.so")

_c = ctypes
_u32p = _c.POINTER(_c.c_uint32)
_u64p = _c.POINTER(_c.c_uint64)
_vpp = _c.POINTER(_c.c_void_p)

# name -> (restype, argtypes); the single source of truth for the binding and for tests/test_abi.py
ABI = {
    "zstdb200_create": (_c.c_int, [_c.POINTER(_c.c_void_p), _c.POINTER(_c.c_int), _c.c_int, _c.c_size_t]),
    "zstdb200_destroy": (None, [_c.c_void_p]),
    "zstdb200_last_error": (_c.c_char_p, [_c.c_void_p]),
    "zstdb200_get_decompressed_size": (_c.c_uint64, [_c.c_void_p, _c.c_uint32]),
    "zstdb200_is_error": (_c.c_int, [_c.c_uint32]),
    "zstdb200_decompress": (_c.c_uint32, [_c.c_void_p, _c.c_void_p, _c.c_uint32, _c.c_void_p, _c.c_uint32]),
    "zstdb200_load_dictionary": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_uint32]),
    "zstdb200_decompress_batch": (_c.c_int, [_c.c_void_p, _vpp, _u32p, _vpp, _u32p, _u32p, _c.c_size_t]),
    "zstdb200_decompress_batch_device": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p,
                                                    _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p]),
    "zstdb200_compress_bound": (_c.c_size_t, [_c.c_size_t]),
    "zstdb200_compress": (_c.c_uint32, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_uint32, _c.c_void_p, _c.c_uint32]),
    "zstdb200_compress_batch": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _vpp, _u32p, _vpp, _u32p, _u32p, _c.c_size_t]),
    "zstdb200_compress_batch_device": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p,
                                                  _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p]),
    "zstdb200_compress_using_dict": (_c.c_uint32, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_uint32, _c.c_void_p, _c.c_uint32]),
    "zstdb200_compress_batch_using_dict": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _vpp, _u32p, _vpp, _u32p, _u32p, _c.c_size_t]),
    "zstdb200_compress_batch_device_using_dict": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p,
                                                             _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p,
                                                             _c.c_size_t, _c.c_void_p]),
    "zstdb200_host_alloc": (_c.c_void_p, [_c.c_size_t]),
    "zstdb200_host_free": (None, [_c.c_void_p]),
    "zstdb200_max_items": (_c.c_size_t, [_c.c_void_p]),
    "zstdb200_device_count": (_c.c_int, [_c.c_void_p]),
    "zstdb200_kernel_launches": (_c.c_uint64, [_c.c_void_p]),
    "zstdb200_version": (_c.c_char_p, []),
    "zstdb200_decompress_batch_device_timed": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p,
                                                          _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p,
                                                          _c.POINTER(_c.c_float), _c.c_int]),
    "zstdb200_decode_kernel_name": (_c.c_char_p, [_c.c_int]),
    "zstdb200_compress_batch_device_timed": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p,
                                                        _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p,
                                                        _c.POINTER(_c.c_float), _c.c_int]),
    "zstdb200_encode_kernel_name": (_c.c_char_p, [_c.c_int]),
    "zstdb200_train_dictionary": (_c.c_uint32, [_c.c_void_p, _c.c_void_p, _c.c_uint32, _c.c_void_p, _u32p, _c.c_size_t, _c.c_void_p]),
    "zstdb200_seekable_info_get": (_c.c_uint32, [_c.c_void_p, _c.c_uint64, _c.c_void_p]),
    "zstdb200_seekable_bound": (_c.c_uint64, [_c.c_uint64, _c.c_uint32]),
    "zstdb200_compress_seekable": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_uint32, _c.c_void_p, _c.c_uint64, _c.c_void_p,
                                              _c.c_uint64, _u64p]),
    "zstdb200_compress_seekable_device": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_uint32, _c.c_void_p, _c.c_uint64,
                                                     _c.c_void_p, _c.c_uint64, _c.c_void_p, _c.c_void_p]),
    "zstdb200_decompress_seekable": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_uint64, _c.c_uint64, _c.c_void_p, _c.c_uint64, _u32p]),
    "zstdb200_decompress_seekable_device": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_uint64, _c.c_uint64, _c.c_void_p,
                                                       _c.c_uint64, _c.c_void_p, _c.c_void_p]),
}


class SeekableInfo(_c.Structure):
    """zstdb200_seekable_info (include/zstdb200.h)."""
    _fields_ = [("content_size", _c.c_uint64), ("data_size", _c.c_uint64), ("n_frames", _c.c_uint32), ("checksums", _c.c_uint32),
                ("max_frame_content", _c.c_uint32), ("max_frame_compressed", _c.c_uint32)]


class SeekableError(RuntimeError):
    """A seekable archive's table or a frame of the decoded range failed (.code, in the library's encoding)."""

    def __init__(self, code, message):
        super().__init__(message)
        self.code = code


class TrainParams(_c.Structure):
    """zstdb200_train_params (include/zstdb200.h); zero fields take the library's defaults."""
    _fields_ = [("k", _c.c_uint32), ("d", _c.c_uint32), ("f", _c.c_uint32), ("accel", _c.c_uint32), ("split_percent", _c.c_uint32),
                ("level", _c.c_int), ("dict_id", _c.c_uint32)]


class TrainError(RuntimeError):
    """zstdb200_train_dictionary returned an error code (.code, in the library's encoding)."""

    def __init__(self, code, message):
        super().__init__(message)
        self.code = code

_lib = None


def load_library():
    """Loads libzstdb200.so (built by zstandard_b200/build.py).  Raises if it is missing: no fallback exists."""
    global _lib
    if _lib is None:
        path = os.environ.get("ZSTDB200_LIB") or LIB_PATH      # development aid: a variant build (zstandard_b200/build.py --debug)
        if not os.path.exists(path):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -m zstandard_b200.build` (nvcc, sm_100a). "
                               "zstandard_b200 has no CPU implementation.")
        lib = ctypes.CDLL(path)
        for name, (res, args) in ABI.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


ERROR_NAMES = {1: "GENERIC", 10: "prefix_unknown", 14: "frameParameter_unsupported", 16: "frameParameter_windowTooLarge",
               20: "corruption_detected", 22: "checksum_wrong", 30: "dictionary_corrupted", 32: "dictionary_wrong",
               44: "tableLog_tooLarge", 46: "maxSymbolValue_tooLarge", 48: "maxSymbolValue_tooSmall", 66: "workSpace_tooSmall",
               70: "dstSize_tooSmall", 72: "srcSize_wrong"}


def is_error(code):
    """ZStdErrors.IsError (csharp/src/ZStdErrors.cs:97-100)."""
    return int(code) > ((-120) & 0xFFFFFFFF)


def error_name(code):
    return ERROR_NAMES.get((-int(code)) & 0xFFFFFFFF, "unknown") if is_error(code) else "no_error"


def _as_u8(buf, writable=False):
    """Zero-copy uint8 view of bytes / bytearray / numpy input (read-only inputs are viewed, not copied).
    A source that is not contiguous is copied; a destination must be written in place, so a non-contiguous (or
    read-only) destination is an error rather than a silent copy that the caller never sees."""
    if isinstance(buf, np.ndarray):
        if writable:
            if not buf.flags.c_contiguous:
                raise ValueError("destination buffers must be C-contiguous")
            if not buf.flags.writeable:
                raise ValueError("destination buffers must be writable")
            return buf.view(np.uint8).reshape(-1)
        return np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
    return np.frombuffer(buf, dtype=np.uint8)


class Context:
    """Owns a zstdb200_ctx (device arenas, streams, staging).  One per caller thread."""

    def __init__(self, devices=None, max_batch_bytes=256 << 20):
        lib = load_library()
        self._lib = lib
        self._h = _c.c_void_p()
        if devices:
            arr = (_c.c_int * len(devices))(*devices)
            rc = lib.zstdb200_create(_c.byref(self._h), arr, len(devices), max_batch_bytes)
        else:
            rc = lib.zstdb200_create(_c.byref(self._h), None, 0, max_batch_bytes)
        if rc != 0:
            self._h = None
            raise RuntimeError(f"zstdb200_create failed (rc={rc}): a CUDA device (B200, sm_100a) is required; "
                               "there is no CPU fallback")
        self.max_batch_bytes = max_batch_bytes

    def close(self):
        if getattr(self, "_h", None):
            self._lib.zstdb200_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def handle(self):
        return self._h

    @property
    def kernel_launches(self):
        return self._lib.zstdb200_kernel_launches(self._h)

    @property
    def device_count(self):
        return self._lib.zstdb200_device_count(self._h)

    @property
    def max_items(self):
        return self._lib.zstdb200_max_items(self._h)

    def last_error(self):
        return self._lib.zstdb200_last_error(self._h).decode()

    def _check(self, name, rc):
        if rc != 0:
            raise RuntimeError(name + " failed: " + self.last_error())

    def _timed(self, name, kernel_name, *args):
        """Runs the *_timed entry point `name` -> {kernel name: ms}."""
        ms = (_c.c_float * 8)()
        self._check(name, getattr(self._lib, name)(self._h, *args, ms, 8))
        names = [kernel_name(k).decode() for k in range(8)]
        return {n: ms[k] for k, n in enumerate(names) if n}

    # ---- host-pointer batches -------------------------------------------------------------------
    def _batch(self, fn, pre, srcs, dsts):
        n = len(srcs)
        sv = [_as_u8(s) for s in srcs]
        dv = [_as_u8(d, writable=True) for d in dsts]
        sp = (_c.c_void_p * n)(*[v.ctypes.data if v.size else None for v in sv])
        dp = (_c.c_void_p * n)(*[v.ctypes.data if v.size else None for v in dv])
        ss = np.array([v.size for v in sv], dtype=np.uint32)
        dc = np.array([v.size for v in dv], dtype=np.uint32)
        res = np.zeros(n, dtype=np.uint32)
        rc = fn(self._h, *pre, sp, ss.ctypes.data_as(_u32p), dp, dc.ctypes.data_as(_u32p), res.ctypes.data_as(_u32p), n)
        if rc != 0:
            raise RuntimeError("zstdb200 batch failed: " + self.last_error())
        return res

    def load_dictionary(self, dictionary):
        """ZSTD_decompress_usingDict (ZStdDecompress.cs:2162-2167, :2366-2475): later decompress calls start every data frame
        from this dictionary, and the *_using_dict compress calls compress against it; None / b"" removes it."""
        d = bytes(dictionary) if dictionary else b""
        self._check("zstdb200_load_dictionary", self._lib.zstdb200_load_dictionary(self._h, d if d else None, len(d)))

    def train_dictionary(self, samples, capacity, **params):
        """Builds a dictionary of at most `capacity` bytes from the sample messages (a list of bytes-like objects) on the
        context's first device; params are the fields of zstdb200_train_params (k, d, f, accel, split_percent, level, dict_id).
        Returns the dictionary bytes; the k and d used are in self.last_train_params.  Raises TrainError on an error result."""
        p = TrainParams(**{k: int(v) for k, v in params.items()})
        views = [_as_u8(s) for s in samples]
        blob = np.concatenate(views) if views else np.zeros(0, dtype=np.uint8)
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        sizes = np.array([v.size for v in views], dtype=np.uint32)
        out = np.zeros(max(int(capacity), 1), dtype=np.uint8)
        r = int(self._lib.zstdb200_train_dictionary(self._h, out.ctypes.data, int(capacity), blob.ctypes.data if blob.size else None,
                                                    sizes.ctypes.data_as(_u32p), len(views), _c.byref(p)))
        if is_error(r):
            raise TrainError(r, f"zstdb200_train_dictionary failed: {error_name(r)} {self.last_error()}".rstrip())
        self.last_train_params = p
        return out[:r].tobytes()

    def decompress_batch(self, srcs, dsts):
        """Decodes srcs[i] into the writable buffer dsts[i]; returns np.uint32 result codes (reference convention)."""
        return self._batch(self._lib.zstdb200_decompress_batch, (), srcs, dsts)

    def compress_batch(self, srcs, dsts, level=3, checksum=True):
        """One zstd frame of srcs[i] into the writable buffer dsts[i]; returns np.uint32 result codes.  level: 1..3, or -7..-1
        (libzstd's fast negative levels: faster and larger, literals stored raw); any other level raises."""
        return self._batch(self._lib.zstdb200_compress_batch, (int(level), 1 if checksum else 0), srcs, dsts)

    def compress_batch_using_dict(self, srcs, dsts, level=3, checksum=True):
        """compress_batch with the dictionary of load_dictionary (raises when none is loaded); the same levels."""
        return self._batch(self._lib.zstdb200_compress_batch_using_dict, (int(level), 1 if checksum else 0), srcs, dsts)

    # ---- seekable archives (zstd's seekable format) ----------------------------------------------
    @staticmethod
    def seekable_bound(size, frame_size):
        """Largest archive compress_seekable writes for `size` bytes in frames of `frame_size`."""
        return int(load_library().zstdb200_seekable_bound(int(size), int(frame_size)))

    def compress_seekable(self, data, frame_size, level=3, checksum=True):
        """One seekable archive of `data`: frames of `frame_size` bytes (each what compress_batch writes for its chunk) and
        the seek table.  Returns bytes; raises on a batch-level failure."""
        sv = _as_u8(data)
        out = np.empty(max(self.seekable_bound(sv.size, frame_size), 1), dtype=np.uint8)
        size = _c.c_uint64(0)
        self._check("zstdb200_compress_seekable", self._lib.zstdb200_compress_seekable(
            self._h, int(level), 1 if checksum else 0, int(frame_size), sv.ctypes.data if sv.size else None, sv.size, out.ctypes.data,
            out.size, _c.byref(size)))
        return out[:size.value].tobytes()

    def seekable_info(self, archive):
        """The archive's table summary (SeekableInfo); raises SeekableError on a malformed table."""
        v = _as_u8(archive)
        info = SeekableInfo()
        r = int(self._lib.zstdb200_seekable_info_get(v.ctypes.data if v.size else None, v.size, _c.byref(info)))
        if r:
            raise SeekableError(r, "seekable table: " + error_name(r))
        return info

    def decompress_seekable(self, archive, offset=0, length=None, out=None):
        """Content bytes [offset, offset + length) of the archive (length None: to the end).  Returns bytes, or fills the
        writable buffer `out` of `length` bytes and returns it.  Raises SeekableError with the first error's code."""
        v = _as_u8(archive)
        if length is None:
            length = max(int(self.seekable_info(v).content_size) - int(offset), 0)
        dv = _as_u8(out, writable=True) if out is not None else np.empty(int(length), dtype=np.uint8)
        if dv.size < length:
            raise ValueError("out is smaller than length")
        code = _c.c_uint32(0)
        self._check("zstdb200_decompress_seekable", self._lib.zstdb200_decompress_seekable(
            self._h, dv.ctypes.data if dv.size else None, int(offset), int(length), v.ctypes.data if v.size else None, v.size,
            _c.byref(code)))
        if code.value:
            raise SeekableError(code.value, f"decompress_seekable: {error_name(code.value)}")
        return out if out is not None else dv.tobytes()

    def compress_seekable_device(self, level, checksum, frame_size, src, size, dst, capacity, dst_size, stream=0, device_index=0):
        """Device pointers: src (size bytes, readable 8 bytes past the end) -> archive at dst; its size to the u64 at dst_size."""
        self._check("zstdb200_compress_seekable_device", self._lib.zstdb200_compress_seekable_device(
            self._h, device_index, int(level), 1 if checksum else 0, int(frame_size), src, int(size), dst, int(capacity), dst_size, stream))

    def decompress_seekable_device(self, dst, offset, length, src, size, code, stream=0, device_index=0):
        """Device pointers: content bytes [offset, offset + length) of the archive src (size bytes) to dst; the u32 at code gets 0
        or the first error."""
        self._check("zstdb200_decompress_seekable_device", self._lib.zstdb200_decompress_seekable_device(
            self._h, device_index, dst, int(offset), int(length), src, int(size), code, stream))

    # ---- device-pointer batches (raw addresses, e.g. torch .data_ptr()) -----------------------
    def decompress_batch_device(self, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream=0, device_index=0):
        self._check("zstdb200_decompress_batch_device", self._lib.zstdb200_decompress_batch_device(
            self._h, device_index, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream))

    def decompress_batch_device_timed(self, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream=0, device_index=0):
        """-> {kernel name: ms} for one synchronised run of the device pipeline."""
        return self._timed("zstdb200_decompress_batch_device_timed", self._lib.zstdb200_decode_kernel_name, device_index, src_base,
                           src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream)

    def compress_batch_device(self, level, checksum, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream=0,
                              device_index=0):
        self._check("zstdb200_compress_batch_device", self._lib.zstdb200_compress_batch_device(
            self._h, device_index, int(level), 1 if checksum else 0, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream))

    def compress_batch_device_using_dict(self, level, checksum, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n,
                                         stream=0, device_index=0):
        """compress_batch_device with the dictionary of load_dictionary (raises when none is loaded)."""
        self._check("zstdb200_compress_batch_device_using_dict", self._lib.zstdb200_compress_batch_device_using_dict(
            self._h, device_index, int(level), 1 if checksum else 0, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream))

    def compress_batch_device_timed(self, level, checksum, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream=0,
                                    device_index=0):
        """-> {kernel name: ms} for one synchronised run of the device pipeline."""
        return self._timed("zstdb200_compress_batch_device_timed", self._lib.zstdb200_encode_kernel_name, device_index, int(level),
                           1 if checksum else 0, src_base, src_off, src_size, dst_base, dst_off, dst_cap, result, n, stream)


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context()
    return _default_ctx


class ZStdDecompress:
    """Mirror of `EPAM.Deltix.ZStd.ZStdDecompress` (csharp/src/ZStdDecompress.cs:37-42): static methods, raw
    `uint` results in the reference's encoding.  `Decompress(dst, src)` and
    `Decompress(dst, dstCapacity, src, srcSize)` follow :2182-2191; `GetDecompressedSize` follows :590-607.
    `DecompressBatch` is the batched-span overload added by this project."""

    @staticmethod
    def GetDecompressedSize(src, srcSize=None):
        v = _as_u8(src)
        n = v.size if srcSize is None else int(srcSize)
        return int(load_library().zstdb200_get_decompressed_size(v.ctypes.data if v.size else None, n))

    @staticmethod
    def Decompress(dst, *args):
        if len(args) == 1:
            src = args[0]
            dv, sv = _as_u8(dst, writable=True), _as_u8(src)
            cap, n = dv.size, sv.size
        elif len(args) == 3:
            cap, src, n = args
            dv, sv = _as_u8(dst, writable=True), _as_u8(src)
        else:
            raise TypeError("Decompress(dst, src) or Decompress(dst, dstCapacity, src, srcSize)")
        ctx = default_context()
        return int(load_library().zstdb200_decompress(ctx.handle, dv.ctypes.data if dv.size else None, int(cap),
                                                      sv.ctypes.data if sv.size else None, int(n)))

    @staticmethod
    def DecompressBatch(srcs, dsts, ctx=None):
        return (ctx or default_context()).decompress_batch(srcs, dsts)


class ZstdDecompressor:
    """Mirror of the reference's Java class `com.epam.deltix.zstd.ZstdDecompressor`
    (java/src/main/java/com/epam/deltix/zstd/ZstdDecompressor.java:18-34) over the same C ABI — what the JNI binding in
    bindings/java/ does on a box with a JDK.  `decompress` returns the bytes written and raises RuntimeError where the
    reference throws (Util.java:32-40); `maxOutputLength == 0` returns 0 without looking at the input
    (ZstdFrameDecompressor.java:164-166).  `getDecompressedSize` follows ZstdFrameDecompressor.java:922-940: RuntimeError
    on a bad magic number, -1 when the header carries no content size.  The decoding itself follows the C# reference
    (the Java port is a second statement of the same format with a few extra restrictions, SURVEY.md §2.2)."""

    def __init__(self, ctx=None):
        self._ctx = ctx

    def decompress(self, input, inputOffset, inputLength, output, outputOffset, maxOutputLength):
        if maxOutputLength == 0:
            return 0
        sv, dv = _as_u8(input), _as_u8(output, writable=True)
        if inputOffset < 0 or inputLength < 0 or inputOffset + inputLength > sv.size or outputOffset < 0 or maxOutputLength < 0 \
                or outputOffset + maxOutputLength > dv.size:
            raise IndexError("offset / length outside the array")
        ctx = self._ctx or default_context()
        r = int(load_library().zstdb200_decompress(ctx.handle, dv.ctypes.data + outputOffset, int(maxOutputLength),
                                                   (sv.ctypes.data + inputOffset) if inputLength else None, int(inputLength)))
        if is_error(r):
            raise RuntimeError("%s: offset=%d" % (error_name(r), inputOffset))
        return r

    def decompressBatch(self, inputs, outputs):
        """[(array, offset, length)] x [(array, offset, maxOutputLength)] -> result codes (one bad frame does not fail the batch)."""
        srcs = [_as_u8(a)[o:o + n] for a, o, n in inputs]
        dsts = [_as_u8(a, writable=True)[o:o + n] for a, o, n in outputs]
        return (self._ctx or default_context()).decompress_batch(srcs, dsts)

    @staticmethod
    def getDecompressedSize(input, offset, length):
        v = _as_u8(input)
        if length < 4 or offset < 0 or offset + length > v.size:
            raise RuntimeError("Not enough input bytes: offset=%d" % offset)
        head = v[offset:offset + min(length, 18)]
        magic = int.from_bytes(head[:4].tobytes(), "little")
        if magic != 0xFD2FB528:
            raise RuntimeError("Invalid magic prefix: %x: offset=%d" % (magic, offset))
        if head.size >= 5 and (int(head[4]) >> 6) == 0 and not (int(head[4]) & 0x20):
            return -1
        return int(load_library().zstdb200_get_decompressed_size(head.ctypes.data, head.size))


class ZStdCompress:
    """Compressor added by this project (the reference has none, SURVEY.md §0 F1); same calling shape."""

    @staticmethod
    def CompressBound(srcSize):
        return int(load_library().zstdb200_compress_bound(int(srcSize)))

    @staticmethod
    def Compress(dst, src, level=3, checksum=True):
        """One frame into dst; the frame size or an error code (GENERIC for a level outside 1..3 and -7..-1)."""
        dv, sv = _as_u8(dst, writable=True), _as_u8(src)
        ctx = default_context()
        return int(load_library().zstdb200_compress(ctx.handle, int(level), 1 if checksum else 0, dv.ctypes.data if dv.size else None,
                                                    dv.size, sv.ctypes.data if sv.size else None, sv.size))

    @staticmethod
    def CompressBatch(srcs, dsts, level=3, checksum=True, ctx=None):
        return (ctx or default_context()).compress_batch(srcs, dsts, level, checksum)

    @staticmethod
    def CompressUsingDict(dst, src, level=3, checksum=True, ctx=None):
        """Compress with the dictionary loaded into the context (Context.load_dictionary); GENERIC when none is."""
        dv, sv = _as_u8(dst, writable=True), _as_u8(src)
        ctx = ctx or default_context()
        return int(load_library().zstdb200_compress_using_dict(ctx.handle, int(level), 1 if checksum else 0, dv.ctypes.data if dv.size else None,
                                                               dv.size, sv.ctypes.data if sv.size else None, sv.size))

    @staticmethod
    def CompressBatchUsingDict(srcs, dsts, level=3, checksum=True, ctx=None):
        return (ctx or default_context()).compress_batch_using_dict(srcs, dsts, level, checksum)


def train_dictionary(samples, capacity, ctx=None, **params):
    """Context.train_dictionary on `ctx` (default: the module's context)."""
    return (ctx or default_context()).train_dictionary(samples, capacity, **params)
