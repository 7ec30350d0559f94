"""Dictionary compression (zstdb200_compress*_using_dict): frames that match against the context's dictionary, start from its
repeat offsets and name its id.  No reference counterpart exists (the reference ships no compressor), so frames are held to
the oracle's ZSTD_decompress_usingDict and to libzstd 1.5.5's, and the ratio to libzstd's ZSTD_CCtx_loadDictionary at the
same level.  CPU tests run the emulation of the dictionary kernels (tests/hostsim/dict_encoder.cpp: the lock-step match stage
and the serial entropy stage) with the encoder dictionary the library prepares (zb_encode.cuh enc_dict_prepare); GPU tests hold
the kernels to it byte for byte."""
import collections
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import helpers

SIZES = [0, 1, 63, 64, 4096, 70000, 131073, 300000]


@pytest.fixture(scope="module")
def material():
    """The log corpus, a 32 KiB trained dictionary, a 30 000-byte raw-content dictionary, and the trained one with its repeat
    offsets edited to 2, 9, 17 (as test_dictionary.py's _material: training on the first 3 MiB)."""
    from tools import corpus, zstd_ref
    log, tick = corpus.log(6 << 20).tobytes(), corpus.tick(2 << 20).tobytes()
    trained = zstd_ref.train_dict([log[i:i + 4096] for i in range(0, 3 << 20, 4096)], 32768)
    raw = log[:30000]
    return {"log": log, "tick": tick, "trained": trained, "raw": raw}


@pytest.fixture(scope="module")
def dictsim():
    """g++ build of tests/hostsim/dict_encoder.cpp (with the __host__ __device__ code it includes)."""
    d = os.path.join(helpers.ROOT, "tests", "hostsim")
    path = os.path.join(d, "_build", "libhostsim_dict.so")
    deps = [os.path.join(d, "dict_encoder.cpp"), os.path.join(d, "serial_encoder.h")] + [
        os.path.join(helpers.ROOT, "zstandard_b200", "csrc", f) for f in ("zb_common.cuh", "zb_format.cuh", "zb_encode.cuh")]
    if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(x) for x in deps):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-static-libstdc++", "-static-libgcc",
                        "-o", path, deps[0]], check=True)
    lib = ctypes.CDLL(path)
    lib.hsdict_set.argtypes = [ctypes.c_char_p, ctypes.c_uint32]
    lib.hsdict_content_offset.restype = ctypes.c_uint32
    lib.hsdict_compress.restype = ctypes.c_uint32
    lib.hsdict_compress.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, ctypes.c_uint32]
    yield lib
    lib.hsdict_set(None, 0)


def _edited(dictsim, trained):
    dictsim.hsdict_set(trained, len(trained))
    at = dictsim.hsdict_content_offset()
    dictsim.hsdict_set(None, 0)
    e = bytearray(trained)
    e[at - 12:at] = b"".join(v.to_bytes(4, "little") for v in (2, 9, 17))
    return bytes(e)


@pytest.fixture(scope="module")
def dicts(dictsim, material):
    return {"trained": material["trained"], "raw": material["raw"], "edited": _edited(dictsim, material["trained"])}


@pytest.fixture(scope="module")
def emu(hostsim, dictsim, oracle):
    """Frames of the dictionary emulation (use_dict, the dictionary of dictsim.hsdict_set) or of hostsim.cpp's emulation of the
    kernels without a dictionary."""
    lib = hostsim.lib
    lib.hostsim_compress_warp2.restype = ctypes.c_uint32
    lib.hostsim_compress_warp2.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, ctypes.c_uint32]

    def compress(data, level, checksum=False, batch_max=None, use_dict=True):
        """-> (result code, frame); the checksum the GPU's k_enc_xxh appends comes from the oracle's XXH64 here."""
        data = bytes(data)
        cap = len(data) + len(data) // 128 + 128
        buf = ctypes.create_string_buffer(cap)
        fn = dictsim.hsdict_compress if use_dict else lib.hostsim_compress_warp2
        r = fn(buf, cap, data, len(data), level, 1 if checksum else 0, len(data) if batch_max is None else batch_max)
        if helpers.is_err(r):
            return r, None
        f = buf.raw[:r]
        if checksum:
            f += (oracle.xxh64(data) & 0xFFFFFFFF).to_bytes(4, "little")
        return len(f), f
    return compress


def _dict_oracle(oracle):
    lib = oracle.lib
    lib.oracle_decompress_using_dict.restype = ctypes.c_uint32
    lib.oracle_decompress_using_dict.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32]

    def run(frame, cap, dictionary):
        buf = ctypes.create_string_buffer(max(cap, 1) + 8)
        r = lib.oracle_decompress_using_dict(buf, cap, frame, len(frame), dictionary, len(dictionary))
        return r, (buf.raw[:r] if not helpers.is_err(r) else None)
    return run


def _frame_dict_id(frame):
    did = frame[4] & 3
    n = [0, 1, 2, 4][did]
    return int.from_bytes(frame[5:5 + n], "little") if n else 0


def _payloads(material, seed=3):
    """Inputs of every size in SIZES from after the training region (log text; every third one tick records)."""
    import random
    rng = random.Random(seed)
    out = []
    for k, n in enumerate(SIZES):
        src = material["tick"] if k % 3 == 2 else material["log"]
        lo = (3 << 20) if src is material["log"] else 0
        i = rng.randrange(lo, len(src) - n)
        out.append(src[i:i + n])
    return out


def test_emulated_frames_decode_with_their_dictionary(dictsim, emu, dicts, material, oracle):
    from tools import zstd_ref
    run = _dict_oracle(oracle)
    trained_id = int.from_bytes(dicts["trained"][4:8], "little")
    payloads = _payloads(material) + _messages(material, "log", 24)
    used, modes = 0, collections.Counter()
    for name, d in dicts.items():
        dictsim.hsdict_set(d, len(d))
        for level in (1, 2, 3):
            for checksum in (False, True):
                for data in payloads:
                    r, f = emu(data, level, checksum)
                    assert f is not None, (name, level, len(data), hex(r))
                    ro, out = run(f, len(data), d)
                    assert ro == len(data) and out == data, (name, level, checksum, len(data), hex(ro))
                    assert zstd_ref.decompress_with_dict(f, len(data), d) == data, (name, level, checksum, len(data))
                    assert _frame_dict_id(f) == (0 if name == "raw" else trained_id)
                    m = helpers.frame_modes(f)
                    modes[name, "treeless"] += sum(v for k, v in m.items() if k[0] == "lit" and k[1] == 3)
                    modes[name, "repeat"] += sum(v for k, v in m.items() if k[0] in ("LL", "OF", "ML") and k[1] == 3)
                    if name != "raw":
                        assert oracle.decompress(f, len(data))[0] == helpers.err(32)       # dictionary_wrong without it
                    else:
                        used += oracle.decompress(f, len(data))[0] != len(data)           # frames that need the content
    assert used > 10
    # the first block reuses an entropy dictionary's tables where that is cheaper; a raw-content dictionary has none
    assert modes["trained", "treeless"] > 20 and modes["trained", "repeat"] > 20 and modes["edited", "repeat"] > 20, modes
    assert modes["raw", "treeless"] == modes["raw", "repeat"] == 0


def test_emulation_starts_from_the_dictionarys_repeat_offsets(dictsim, emu, dicts, material, oracle):
    """The edited dictionary's repeat offsets (2, 9, 17) differ from the default 1, 4, 8.  A message that starts with a run of
    one byte value is matched at once with the first repeat offset (repeat code 1, before any offset of the frame replaced
    it): it only decodes if the encoder started from the dictionary's offsets, as the decoders do (an encoder that keeps
    1 and 4 fails on almost all of these)."""
    from tools import zstd_ref
    run = _dict_oracle(oracle)
    d = dicts["edited"]
    dictsim.hsdict_set(d, len(d))
    log = material["log"]
    for level in (1, 2, 3):
        for k in range(64):
            o = (4 << 20) + 997 * k
            data = bytes([0x21 + k % 90]) * (6 + k % 20) + log[o:o + 3000]
            r, f = emu(data, level)
            assert zstd_ref.decompress_with_dict(f, len(data), d) == data, (level, k)
            assert run(f, len(data), d) == (len(data), data), (level, k)


def _run_starts(material, count=16):
    """Messages that start with a run of one byte value: matched at once with the frame's first repeat offset."""
    log = material["log"]
    return [bytes([0x21 + k]) * (6 + k) + log[(5 << 20) + 1013 * k:(5 << 20) + 1013 * k + 3000] for k in range(count)]


def _messages(material, kind, count=256):
    src = material[kind]
    base = (3 << 20) if kind == "log" else (1 << 20)
    return [src[base + 4096 * k:base + 4096 * (k + 1)] for k in range(count)]


@pytest.mark.parametrize("kind", ["log", "tick"])
def test_emulated_ratio_band_against_libzstd(dictsim, emu, dicts, material, kind):
    """4 KiB messages: total size within 3 % of libzstd's with the same dictionary and level (no checksum either side); on log
    text with the trained dictionary at least 15 % smaller than without a dictionary."""
    from tools import zstd_ref
    msgs = _messages(material, kind)
    for name in ("trained", "raw"):
        d = dicts[name]
        dictsim.hsdict_set(d, len(d))
        for level in (1, 2, 3):
            ours = sum(emu(m, level)[0] for m in msgs)
            ref = sum(len(zstd_ref.compress_with_dict(m, d, level, False)) for m in msgs)
            assert ours <= ref * 1.03, (kind, name, level, ours, ref)
            if kind == "log" and name == "trained":
                plain = sum(emu(m, level, use_dict=False)[0] for m in msgs)
                assert ours <= plain * 0.85, (level, ours, plain)


def test_malformed_dictionary_and_no_dictionary(dictsim, emu, dicts):
    broken = bytearray(dicts["trained"]); broken[8:40] = bytes(32)
    dictsim.hsdict_set(bytes(broken), len(broken))
    assert emu(b"x" * 5000, 1)[0] == helpers.err(30)                        # dictionary_corrupted, as on the decode side
    dictsim.hsdict_set(None, 0)
    assert emu(b"x" * 5000, 1)[0] == helpers.err(1)


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
def _gpu_compress(ctx, payloads, level, checksum=False, use_dict=True):
    import zstandard_b200 as zb
    dsts = [np.zeros(max(zb.ZStdCompress.CompressBound(len(p)), 1), dtype=np.uint8) for p in payloads]
    fn = ctx.compress_batch_using_dict if use_dict else ctx.compress_batch
    res = fn(payloads, dsts, level=level, checksum=checksum)
    return [d[:int(r)].tobytes() if not helpers.is_err(int(r)) else int(r) for r, d in zip(res, dsts)]


@pytest.mark.gpu
def test_gpu_matches_the_emulation_byte_for_byte(gpu_ctx, dictsim, emu, dicts, material):
    payloads = _payloads(material, seed=11) + _payloads(material, seed=12) + _run_starts(material) + _messages(material, "log", 32)
    small = [p for p in payloads if len(p) <= 131072]
    try:
        for name, d in dicts.items():
            gpu_ctx.load_dictionary(d)
            dictsim.hsdict_set(d, len(d))
            for batch in (payloads, small):                  # both table-size regimes (zb_encode.cuh enc_hlog_*)
                biggest = max(len(p) for p in batch)
                for level in (1, 2, 3):
                    got = _gpu_compress(gpu_ctx, batch, level)
                    for p, g in zip(batch, got):
                        assert g == emu(p, level, batch_max=biggest)[1], (name, level, len(p), biggest)
    finally:
        gpu_ctx.load_dictionary(None)


@pytest.mark.gpu
def test_gpu_frames_decode_on_the_same_context(gpu_ctx, dicts, material, oracle):
    from tools import zstd_ref
    run = _dict_oracle(oracle)
    payloads = _payloads(material, seed=21) + _messages(material, "log", 64) + _run_starts(material)
    try:
        for name, d in dicts.items():
            gpu_ctx.load_dictionary(d)
            for level in (1, 2, 3):
                frames = _gpu_compress(gpu_ctx, payloads, level, checksum=True)
                outs = [np.zeros(max(len(p), 1), dtype=np.uint8)[:len(p)] for p in payloads]
                res = gpu_ctx.decompress_batch(frames, outs)
                for p, f, r, o in zip(payloads, frames, res, outs):
                    assert int(r) == len(p) and o.tobytes() == p, (name, level, len(p), hex(int(r)))
                    assert run(f, len(p), d) == (len(p), p)
                    assert zstd_ref.decompress_with_dict(f, len(p), d) == p
    finally:
        gpu_ctx.load_dictionary(None)


@pytest.mark.gpu
def test_gpu_device_pointer_path_matches_the_host_path(gpu_ctx, dicts, material):
    """A host batch of 48 MiB runs in several concurrent slices (shared-memory match tables); the device-pointer call has the
    device to itself (global-memory match tables).  Both write the same bytes."""
    import torch
    import zstandard_b200 as zb
    log = material["log"]
    n, chunk = 12000, 4096
    msgs = [log[(3 << 20) + 257 * k:(3 << 20) + 257 * k + chunk] for k in range(n)]
    bound = (zb.ZStdCompress.CompressBound(chunk) + 15) // 16 * 16
    dev = torch.device("cuda:0")
    t_src = torch.zeros(n * chunk + 64, dtype=torch.uint8, device=dev)
    t_src[:n * chunk] = torch.from_numpy(np.frombuffer(b"".join(msgs), dtype=np.uint8).copy()).to(dev)
    t_dst = torch.zeros(n * bound, dtype=torch.uint8, device=dev)
    t_soff = torch.arange(n, dtype=torch.int64, device=dev) * chunk
    t_doff = torch.arange(n, dtype=torch.int64, device=dev) * bound
    t_ssz = torch.full((n,), chunk, dtype=torch.int32, device=dev)
    t_cap = torch.full((n,), bound, dtype=torch.int32, device=dev)
    t_res = torch.zeros(n, dtype=torch.int32, device=dev)
    try:
        gpu_ctx.load_dictionary(dicts["trained"])
        for level in (1, 2, 3):
            host = _gpu_compress(gpu_ctx, msgs, level, checksum=True)
            torch.cuda.synchronize()
            gpu_ctx.compress_batch_device_using_dict(level, True, t_src.data_ptr(), t_soff.data_ptr(), t_ssz.data_ptr(), t_dst.data_ptr(),
                                                     t_doff.data_ptr(), t_cap.data_ptr(), t_res.data_ptr(), n)
            torch.cuda.synchronize()
            res = t_res.cpu().numpy().view(np.uint32)
            out = t_dst.cpu().numpy()
            for k in range(n):
                assert out[k * bound:k * bound + int(res[k])].tobytes() == host[k], (level, k)
    finally:
        gpu_ctx.load_dictionary(None)


@pytest.mark.gpu
def test_gpu_interface_cases(dicts, material):
    import torch
    import zstandard_b200 as zb
    ctx = zb.Context(max_batch_bytes=16 << 20)
    try:
        payloads = _payloads(material, seed=31)
        with pytest.raises(RuntimeError):
            _gpu_compress(ctx, payloads, 1)                                       # no dictionary loaded
        d1 = torch.zeros(64, dtype=torch.uint8, device="cuda:0")
        with pytest.raises(RuntimeError):
            ctx.compress_batch_device_using_dict(1, False, d1.data_ptr(), d1.data_ptr(), d1.data_ptr(), d1.data_ptr(), d1.data_ptr(),
                                                 d1.data_ptr(), d1.data_ptr(), 1)
        dst = np.zeros(200, dtype=np.uint8)
        assert zb.ZStdCompress.CompressUsingDict(dst, b"x" * 100, 1, ctx=ctx) == helpers.err(1)
        plain = {lv: _gpu_compress(ctx, payloads, lv, use_dict=False) for lv in (1, 3)}
        broken = bytearray(dicts["trained"]); broken[8:40] = bytes(32)
        ctx.load_dictionary(bytes(broken))
        assert all(r == helpers.err(30) for r in _gpu_compress(ctx, payloads, 2))
        ctx.load_dictionary(dicts["trained"])
        tid = int.from_bytes(dicts["trained"][4:8], "little")
        assert all(_frame_dict_id(f) == tid for f in _gpu_compress(ctx, payloads, 2))
        n = zb.ZStdCompress.CompressUsingDict(dst, b"y" * 100, 1, ctx=ctx)
        assert not helpers.is_err(n) and _frame_dict_id(bytes(dst[:n])) == tid
        other = bytearray(dicts["trained"]); other[4:8] = (tid ^ 0x55555555).to_bytes(4, "little")
        ctx.load_dictionary(bytes(other))
        assert all(_frame_dict_id(f) == tid ^ 0x55555555 for f in _gpu_compress(ctx, payloads, 2))
        ctx.load_dictionary(dicts["raw"])
        assert all(_frame_dict_id(f) == 0 for f in _gpu_compress(ctx, payloads, 2))
        for lv in (1, 3):                                                          # the plain calls ignore the dictionary
            assert _gpu_compress(ctx, payloads, lv, use_dict=False) == plain[lv]
    finally:
        ctx.close()


@pytest.mark.gpu
def test_gpu_one_context_over_two_devices(dicts, material):
    import torch
    import zstandard_b200 as zb
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    payloads = _payloads(material, seed=41) + _messages(material, "log", 512)
    one, two = zb.Context(devices=[0], max_batch_bytes=64 << 20), zb.Context(devices=[0, 1], max_batch_bytes=64 << 20)
    try:
        for ctx in (one, two):
            ctx.load_dictionary(dicts["trained"])
        for level in (1, 2, 3):
            assert _gpu_compress(one, payloads, level, checksum=True) == _gpu_compress(two, payloads, level, checksum=True)
    finally:
        one.close(); two.close()
