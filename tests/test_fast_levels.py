"""Compression levels -7..-1: libzstd's fast negative levels (acceleration = -level).  The match stage probes pairs of
adjacent positions with a stride of 1 + acceleration and every compressed block stores its literals raw.  CPU tests run the
lock-step emulation of the kernels at these levels (tests/hostsim/fast_levels.cpp, with and without a dictionary) against the
oracle, libzstd 1.5.5 and libzstd's ratio at the same level; GPU tests hold the kernels to the emulation byte for byte on the
host batch path (shared-memory match tables) and the device-pointer path (global tables)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import helpers

LEVELS = [-1, -2, -3, -4, -5, -6, -7]
SIZES = [0, 1, 63, 64, 4096, 131072, 131073, 1 << 20]


@pytest.fixture(scope="module")
def material():
    from tools import corpus, zstd_ref
    log, tick = corpus.log(24 << 20).tobytes(), corpus.tick(24 << 20).tobytes()
    trained = zstd_ref.train_dict([log[i:i + 4096] for i in range(0, 3 << 20, 4096)], 32768)
    return {"log": log, "tick": tick, "random": corpus.random_(2 << 20).tobytes(), "trained": trained}


@pytest.fixture(scope="module")
def fastsim():
    """g++ build of tests/hostsim/fast_levels.cpp (with dict_encoder.cpp and the __host__ __device__ code they include)."""
    d = os.path.join(helpers.ROOT, "tests", "hostsim")
    path = os.path.join(d, "_build", "libhostsim_fast.so")
    deps = [os.path.join(d, f) for f in ("fast_levels.cpp", "dict_encoder.cpp", "serial_encoder.h")] + [
        os.path.join(helpers.ROOT, "zstandard_b200", "csrc", f) for f in ("zb_common.cuh", "zb_format.cuh", "zb_encode.cuh")]
    if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(x) for x in deps):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-static-libstdc++", "-static-libgcc",
                        "-o", path, deps[0]], check=True)
    lib = ctypes.CDLL(path)
    lib.hsdict_set.argtypes = [ctypes.c_char_p, ctypes.c_uint32]
    lib.hsfast_compress.restype = ctypes.c_uint32
    lib.hsfast_compress.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int,
                                    ctypes.c_uint32, ctypes.c_int]
    yield lib
    lib.hsdict_set(None, 0)


@pytest.fixture(scope="module")
def emu(fastsim, oracle):
    """One frame of the emulation, with the dictionary of fastsim.hsdict_set when use_dict.  batch_max: the largest chunk of the
    call (the match table's size).  The checksum k_enc_xxh appends comes from the oracle's XXH64."""
    def compress(data, level, checksum=False, batch_max=None, use_dict=False):
        data = bytes(data)
        cap = len(data) + len(data) // 128 + 128
        buf = ctypes.create_string_buffer(cap)
        r = fastsim.hsfast_compress(buf, cap, data, len(data), level, 1 if checksum else 0,
                                    len(data) if batch_max is None else batch_max, 1 if use_dict else 0)
        assert not helpers.is_err(r), hex(r)
        f = buf.raw[:r]
        if checksum:
            f += (oracle.xxh64(data) & 0xFFFFFFFF).to_bytes(4, "little")
        return f
    return compress


def _input(material, kind, n, at=0):
    if kind == "constant":
        return b"\x5a" * n
    src = material[kind]
    return src[at:at + n]


def _assert_raw_literals(frame):
    """Every compressed block's literals section is raw (type 0)."""
    modes = helpers.frame_modes(frame)
    lit = {k: v for k, v in modes.items() if k[0] == "lit"}
    assert all(k[1] == 0 for k in lit), modes
    return sum(lit.values())


@pytest.mark.parametrize("level", LEVELS)
def test_round_trips_with_raw_literals(emu, material, oracle, level):
    from tools import zstd_ref
    compressed = 0
    for kind in ("log", "tick", "random", "constant"):
        for n in SIZES:
            data = _input(material, kind, n, at=4096 * (-level))
            for checksum in (False, True):
                f = emu(data, level, checksum)
                ro, out, _ = oracle.decompress(f, len(data))
                assert ro == len(data) and out == data, (kind, n, checksum, hex(ro))
                assert zstd_ref.decompress(f, len(data)) == data, (kind, n, checksum)
                compressed += _assert_raw_literals(f)
    assert compressed > 20


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("kind", ["log", "tick"])
def test_ratio_band_against_libzstd(emu, material, kind, level):
    """Total size at most 1.03 x libzstd's at the same level (no checksum either side), chunks of 4 KiB .. 1 MiB."""
    from tools import zstd_ref
    raw = material[kind]
    for chunk in (4096, 65536, 131072, 1 << 20):
        n = min(256, (16 << 20) // chunk)
        chunks = [raw[i * chunk:(i + 1) * chunk] for i in range(n)]
        ours = sum(len(emu(c, level, batch_max=chunk)) for c in chunks)
        ref = sum(len(zstd_ref.compress(c, level, checksum=False)) for c in chunks)
        assert ours <= ref * 1.03, (kind, chunk, level, ours, ref)


@pytest.mark.parametrize("level", LEVELS)
def test_dictionary_round_trips_and_ratio_band(emu, fastsim, material, oracle, level):
    """4 KiB log messages after the training region with a ZDICT dictionary: frames decode with the dictionary through the oracle
    and libzstd, literals stay raw, and the total is at most 1.03 x libzstd's compress_with_dict at the same level."""
    from tools import zstd_ref
    d = material["trained"]
    fastsim.hsdict_set(d, len(d))
    oracle.lib.oracle_decompress_using_dict.restype = ctypes.c_uint32
    oracle.lib.oracle_decompress_using_dict.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32,
                                                        ctypes.c_char_p, ctypes.c_uint32]
    log = material["log"]
    msgs = [log[(3 << 20) + 4096 * k:(3 << 20) + 4096 * (k + 1)] for k in range(256)]
    ours = 0
    for k, m in enumerate(msgs):
        f = emu(m, level, checksum=k % 2 == 1, use_dict=True)
        ours += len(f) - (4 if k % 2 else 0)
        _assert_raw_literals(f)
        if k % 8 == 0:
            buf = ctypes.create_string_buffer(len(m) + 8)
            assert oracle.lib.oracle_decompress_using_dict(buf, len(m), f, len(f), d, len(d)) == len(m)
            assert buf.raw[:len(m)] == m
            assert zstd_ref.decompress_with_dict(f, len(m), d) == m
    ref = sum(len(zstd_ref.compress_with_dict(m, d, level, False)) for m in msgs)
    assert ours <= ref * 1.03, (level, ours, ref)
    for n in (0, 1, 63, 64, 131073, 300000):                  # other sizes, one block and several
        data = log[(5 << 20):(5 << 20) + n]
        f = emu(data, level, checksum=True, use_dict=True)
        assert zstd_ref.decompress_with_dict(f, len(data), d) == data, n


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
def _payloads(material):
    """Chunks of every size class, above 128 KiB mixed with small ones."""
    import random
    rng = random.Random(5)
    out = []
    for k, n in enumerate([0, 1, 63, 64, 100, 4096, 5000, 65536, 131072, 131073, 200000, 300000, 1 << 20] * 2):
        kind = ("log", "tick", "random", "constant")[k % 4] if k % 7 else "log"
        at = rng.randrange(0, (2 << 20) - n) if kind == "random" else rng.randrange(0, (20 << 20) - n)
        out.append(_input(material, kind, n, at))
    return out


def _gpu(ctx, payloads, level, checksum=False, use_dict=False):
    import zstandard_b200 as zb
    dsts = [np.zeros(max(zb.ZStdCompress.CompressBound(len(p)), 1), dtype=np.uint8) for p in payloads]
    fn = ctx.compress_batch_using_dict if use_dict else ctx.compress_batch
    res = fn(payloads, dsts, level=level, checksum=checksum)
    assert not any(helpers.is_err(int(r)) for r in res)
    return [d[:int(r)].tobytes() for r, d in zip(res, dsts)]


def _device(ctx, payloads, level, use_dict=False):
    """The device-pointer call (global-memory match tables) over payloads laid out back to back."""
    import torch
    import zstandard_b200 as zb
    n = len(payloads)
    src = np.frombuffer(b"".join(payloads) + bytes(64), dtype=np.uint8).copy()
    soff = np.cumsum([0] + [len(p) for p in payloads[:-1]]).astype(np.int64)
    bounds = [(zb.ZStdCompress.CompressBound(len(p)) + 15) // 16 * 16 for p in payloads]
    doff = np.cumsum([0] + bounds[:-1]).astype(np.int64)
    dev = torch.device("cuda:0")
    t_src = torch.from_numpy(src).to(dev)
    t_dst = torch.zeros(sum(bounds), dtype=torch.uint8, device=dev)
    t_soff, t_doff = torch.from_numpy(soff).to(dev), torch.from_numpy(doff).to(dev)
    t_ssz = torch.tensor([len(p) for p in payloads], dtype=torch.int32, device=dev)
    t_cap = torch.tensor(bounds, dtype=torch.int32, device=dev)
    t_res = torch.zeros(n, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    fn = ctx.compress_batch_device_using_dict if use_dict else ctx.compress_batch_device
    fn(level, False, t_src.data_ptr(), t_soff.data_ptr(), t_ssz.data_ptr(), t_dst.data_ptr(), t_doff.data_ptr(), t_cap.data_ptr(),
       t_res.data_ptr(), n)
    torch.cuda.synchronize()
    res = t_res.cpu().numpy().view(np.uint32)
    out = t_dst.cpu().numpy()
    assert not any(helpers.is_err(int(r)) for r in res)
    return [out[doff[k]:doff[k] + int(res[k])].tobytes() for k in range(n)]


@pytest.mark.gpu
def test_gpu_matches_the_emulation(gpu_ctx, emu, material):
    payloads = _payloads(material)
    small = [p for p in payloads if len(p) <= 131072]
    for level in LEVELS:
        for batch in (payloads, small):                      # both table-size regimes (zb_encode.cuh enc_hlog_*)
            biggest = max(len(p) for p in batch)
            want = [emu(p, level, batch_max=biggest) for p in batch]
            assert _gpu(gpu_ctx, batch, level) == want, (level, biggest)
            assert _device(gpu_ctx, batch, level) == want, (level, biggest)


@pytest.mark.gpu
def test_gpu_matches_the_emulation_with_a_dictionary(gpu_ctx, emu, fastsim, material):
    d = material["trained"]
    log = material["log"]
    msgs = [log[(3 << 20) + 4096 * k:(3 << 20) + 4096 * (k + 1)] for k in range(64)]
    payloads = _payloads(material) + msgs
    small = [p for p in payloads if len(p) <= 131072]
    fastsim.hsdict_set(d, len(d))
    try:
        gpu_ctx.load_dictionary(d)
        for level in LEVELS:
            for batch in (payloads, small):
                biggest = max(len(p) for p in batch)
                want = [emu(p, level, batch_max=biggest, use_dict=True) for p in batch]
                assert _gpu(gpu_ctx, batch, level, use_dict=True) == want, (level, biggest)
                assert _device(gpu_ctx, batch, level, use_dict=True) == want, (level, biggest)
    finally:
        gpu_ctx.load_dictionary(None)


@pytest.mark.gpu
def test_gpu_frames_decode_on_the_same_context(gpu_ctx, material):
    from tools import zstd_ref
    payloads = _payloads(material)
    log = material["log"]
    msgs = [log[(3 << 20) + 4096 * k:(3 << 20) + 4096 * (k + 1)] for k in range(64)]
    d = material["trained"]
    try:
        for use_dict in (False, True):
            gpu_ctx.load_dictionary(d if use_dict else None)
            batch = payloads + (msgs if use_dict else [])
            for level in LEVELS:
                frames = _gpu(gpu_ctx, batch, level, checksum=True, use_dict=use_dict)
                outs = [np.zeros(max(len(p), 1), dtype=np.uint8)[:len(p)] for p in batch]
                res = gpu_ctx.decompress_batch(frames, outs)
                for p, f, r, o in zip(batch, frames, res, outs):
                    assert int(r) == len(p) and o.tobytes() == p, (use_dict, level, len(p), hex(int(r)))
                    _assert_raw_literals(f)
                for p, f in list(zip(batch, frames))[::5]:
                    got = zstd_ref.decompress_with_dict(f, len(p), d) if use_dict else zstd_ref.decompress(f, len(p))
                    assert got == p
    finally:
        gpu_ctx.load_dictionary(None)


@pytest.mark.gpu
def test_gpu_levels_outside_both_ranges_are_rejected(material):
    import torch
    import zstandard_b200 as zb
    ctx = zb.Context(max_batch_bytes=16 << 20)
    msg = "level must be 1..3 or -7..-1"
    try:
        ctx.load_dictionary(material["trained"])
        src = np.frombuffer(material["log"][:5000], dtype=np.uint8)
        dst = np.zeros(zb.ZStdCompress.CompressBound(5000), dtype=np.uint8)
        t = torch.zeros(64, dtype=torch.uint8, device="cuda:0")
        p = t.data_ptr()
        for level in (-8, 0, 4):
            for fn in (ctx.compress_batch, ctx.compress_batch_using_dict):
                with pytest.raises(RuntimeError, match=msg):
                    fn([src], [dst], level=level)
            assert zb.ZStdCompress.CompressUsingDict(dst, src, level, ctx=ctx) == helpers.err(1)
            assert ctx.last_error() == msg
            for fn in (ctx.compress_batch_device, ctx.compress_batch_device_using_dict, ctx.compress_batch_device_timed):
                with pytest.raises(RuntimeError, match=msg):
                    fn(level, False, p, p, p, p, p, p, p, 1)
            dctx = zb.default_context()
            assert zb.ZStdCompress.Compress(dst, src, level) == helpers.err(1)
            assert dctx.last_error() == msg
        for level in (-7, -1, 1, 3):                              # the ends of both ranges are accepted
            r = ctx.compress_batch([src], [dst], level=level)
            assert not helpers.is_err(int(r[0]))
        with pytest.raises(zb.TrainError):                        # the trainer keeps levels 1..3
            ctx.train_dictionary([material["log"][i:i + 4096] for i in range(0, 1 << 20, 4096)], 16384, level=-1)
    finally:
        ctx.close()
