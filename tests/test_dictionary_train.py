"""Dictionary training (zstdb200_train_dictionary): content selected as libzstd 1.5.5's fastCover trainer selects it, entropy
tables from this library's match stage.  CPU tests hold the emulation (tests/hostsim/dict_train.cpp) to ZDICT: the same
selection and id, dictionaries that libzstd and the oracle accept, and a ratio within 3 % of ZDICT_trainFromBuffer's.  GPU tests
hold the library to the emulation byte for byte."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import helpers

CAP = 32768


@pytest.fixture(scope="module")
def trainsim():
    """g++ build of tests/hostsim/dict_train.cpp (it includes dict_encoder.cpp: hsdict_* are exported too)."""
    d = os.path.join(helpers.ROOT, "tests", "hostsim")
    path = os.path.join(d, "_build", "libhostsim_dict_train.so")
    deps = [os.path.join(d, f) for f in ("dict_train.cpp", "dict_encoder.cpp", "serial_encoder.h")] + [
        os.path.join(helpers.ROOT, "zstandard_b200", "csrc", f) for f in ("zb_common.cuh", "zb_format.cuh", "zb_encode.cuh", "zb_dict_train.cuh")]
    if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(x) for x in deps):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-static-libstdc++", "-static-libgcc",
                        "-o", path, deps[0]], check=True)
    lib = ctypes.CDLL(path)
    lib.dtsim_train.restype = ctypes.c_uint32
    lib.dtsim_train.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p]
    lib.hsdict_set.argtypes = [ctypes.c_char_p, ctypes.c_uint32]
    lib.hsdict_content_offset.restype = ctypes.c_uint32
    lib.hsdict_compress.restype = ctypes.c_uint32
    lib.hsdict_compress.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, ctypes.c_uint32]
    return lib


def emu_train(lib, samples, capacity=CAP, **params):
    """-> (result code, dictionary or None, k chosen)"""
    blob = b"".join(samples)
    sizes = (ctypes.c_uint32 * max(len(samples), 1))(*[len(s) for s in samples])
    p = (ctypes.c_uint32 * 7)(*[params.get(k, 0) for k in ("k", "d", "f", "accel", "split_percent", "level", "dict_id")])
    buf = ctypes.create_string_buffer(capacity)
    r = lib.dtsim_train(buf, capacity, blob, sizes, len(samples), p)
    return r, (None if helpers.is_err(r) else buf.raw[:r]), p[0]


# ---- libzstd's trainers through ctypes ----------------------------------------------------------------------------------------
class _ZParams(ctypes.Structure):
    _fields_ = [("compressionLevel", ctypes.c_int), ("notificationLevel", ctypes.c_uint), ("dictID", ctypes.c_uint)]


class _FastCover(ctypes.Structure):
    _fields_ = [("k", ctypes.c_uint), ("d", ctypes.c_uint), ("f", ctypes.c_uint), ("steps", ctypes.c_uint), ("nbThreads", ctypes.c_uint),
                ("splitPoint", ctypes.c_double), ("accel", ctypes.c_uint), ("shrinkDict", ctypes.c_uint),
                ("shrinkDictMaxRegression", ctypes.c_uint), ("zParams", _ZParams)]


def _z():
    from tools import zstd_ref
    z = zstd_ref._Z
    z.ZDICT_trainFromBuffer_fastCover.restype = ctypes.c_size_t
    z.ZDICT_trainFromBuffer_fastCover.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint, _FastCover]
    z.ZDICT_optimizeTrainFromBuffer_fastCover.restype = ctypes.c_size_t
    z.ZDICT_optimizeTrainFromBuffer_fastCover.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint,
                                                          ctypes.POINTER(_FastCover)]
    z.ZDICT_getDictHeaderSize.restype = ctypes.c_size_t
    z.ZDICT_getDictHeaderSize.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
    return z


def zdict_train(samples, capacity=CAP, k=None, d=8, f=20, accel=1, split=None):
    """k given: ZDICT_trainFromBuffer_fastCover (split None) or ZDICT_optimizeTrainFromBuffer_fastCover with k fixed (split
    given); k None: ZDICT_trainFromBuffer.  -> dictionary"""
    from tools import zstd_ref
    if k is None:
        return zstd_ref.train_dict(samples, capacity)
    z = _z()
    blob = b"".join(samples)
    sizes = (ctypes.c_size_t * len(samples))(*[len(s) for s in samples])
    buf = ctypes.create_string_buffer(capacity)
    p = _FastCover(k=k, d=d, f=f, accel=accel, splitPoint=split or 0.0)
    if split is None:
        n = z.ZDICT_trainFromBuffer_fastCover(buf, capacity, blob, sizes, len(samples), p)
    else:
        n = z.ZDICT_optimizeTrainFromBuffer_fastCover(buf, capacity, blob, sizes, len(samples), ctypes.byref(p))
    assert not z.ZDICT_isError(n)
    return buf.raw[:n]


def header_size(dictionary):
    return _z().ZDICT_getDictHeaderSize(dictionary, len(dictionary))


# ---- corpora -------------------------------------------------------------------------------------------------------------------
def log_samples(total, size=4096, base=0):
    from tools import corpus
    text = corpus.log(base + total).tobytes()
    return [text[base + i:base + i + size] for i in range(0, total, size)]


def mixed_samples():
    """1 B .. 64 KiB, some shorter than 8 bytes"""
    import random
    from tools import corpus
    rng = random.Random(5)
    text = corpus.log(4 << 20).tobytes()
    out, pos = [], 0
    while pos < (3 << 20):
        n = rng.choice([1, 3, 7, 8, 100, 1000, 4096, 20000, 65536]) if rng.random() < 0.8 else rng.randrange(1, 65537)
        out.append(text[pos:pos + n]); pos += n
    return out


def tick_samples():
    from tools import corpus
    t = corpus.tick(2 << 20).tobytes()
    return [t[i:i + 4096] for i in range(0, 2 << 20, 4096)]


def repetitive_samples():
    """Few distinct messages: every d-mer is selected long before 32 KiB, then ten epochs in a row score zero"""
    msgs = [(b"user %d logged in from host-%d; session ok\n" % (i, i * 7)) * 3 for i in range(6)]
    return [msgs[i % 6] for i in range(600)]


CONFIGS = {
    "k1024": (lambda: log_samples(3 << 20), dict(k=1024, d=8, f=20, accel=1, split_percent=100), dict(k=1024, d=8, f=20, accel=1)),
    "k200_d6_f18": (lambda: log_samples(3 << 20), dict(k=200, d=6, f=18, accel=1), dict(k=200, d=6, f=18, accel=1)),
    "k1024_accel4": (lambda: log_samples(3 << 20), dict(k=1024, d=8, accel=4), dict(k=1024, d=8, accel=4)),
    "k1511_split75": (lambda: log_samples(3 << 20), dict(k=1511, split_percent=75), dict(k=1511, split=0.75)),
    "mixed": (mixed_samples, dict(k=1024), dict(k=1024)),
    "tick": (tick_samples, dict(k=512), dict(k=512)),
    "repetitive": (repetitive_samples, dict(k=300), dict(k=300)),
}


def _same_selection(ours, theirs):
    a, b = ours[header_size(ours):], theirs[header_size(theirs):]
    short, long_ = (a, b) if len(a) <= len(b) else (b, a)
    return len(short) > 0 and long_.startswith(short) and ours[4:8] == theirs[4:8]


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_emulated_selection_matches_zdict(trainsim, name):
    """libzstd keeps the front of the selection when the header leaves less room: the longer content starts with the shorter.
    Equal selections give equal ids (ZDICT's XXH64 rule over the whole selection)."""
    make, ours_p, theirs_p = CONFIGS[name]
    samples = make()
    r, ours, k = emu_train(trainsim, samples, **ours_p)
    assert ours is not None, hex(r)
    assert k == ours_p["k"]
    theirs = zdict_train(samples, **theirs_p)
    assert _same_selection(ours, theirs), name
    if name == "repetitive":
        assert len(theirs) < CAP // 2 and len(ours) - header_size(ours) == len(theirs) - header_size(theirs)


def test_emulated_dictionaries_are_valid(trainsim, oracle):
    from tools import zstd_ref
    run = helpers.Oracle().lib
    run.oracle_decompress_using_dict.restype = ctypes.c_uint32
    run.oracle_decompress_using_dict.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32]
    held = log_samples(1 << 20, base=4 << 20)[:64]
    good_modes = 0
    for name, (make, ours_p, _) in sorted(CONFIGS.items()):
        r, dic, _ = emu_train(trainsim, make(), **ours_p)
        hs = header_size(dic)
        trainsim.hsdict_set(dic, len(dic))                                  # the library's dict_load
        assert trainsim.hsdict_content_offset() == hs, name
        buf = ctypes.create_string_buffer(8192)
        assert not helpers.is_err(trainsim.hsdict_compress(buf, 8192, held[0], len(held[0]), 1, 0, 4096)), name
        for m in held[:16]:
            f = zstd_ref.compress_with_dict(m, dic, 3, False)               # ZSTD_CCtx_loadDictionary accepts it
            out = ctypes.create_string_buffer(len(m) + 8)
            assert run.oracle_decompress_using_dict(out, len(m), f, len(f), dic, len(dic)) == len(m) and out.raw[:len(m)] == m
            if name == "k1024":
                modes = helpers.frame_modes(f)
                good_modes += any(k[0] == "lit" and k[1] == 3 for k in modes) and any(k[0] in ("LL", "OF", "ML") and k[1] == 3 for k in modes)
    trainsim.hsdict_set(None, 0)
    assert good_modes > 8, good_modes


def test_emulated_ratio_within_three_percent_of_zdict(trainsim):
    """Default parameters, 3 MiB of 4 KiB log samples; 256 held-out messages.  Totals with libzstd level 3 and with the emulated
    encoder at levels 1-3, against ZDICT_trainFromBuffer's dictionary."""
    from tools import zstd_ref
    samples = log_samples(3 << 20)
    held = log_samples(1 << 20, base=4 << 20)
    r, ours, k = emu_train(trainsim, samples)
    assert ours is not None and k in (50, 537, 1024, 1511, 1998)
    theirs = zdict_train(samples)
    ref = lambda d, lv: sum(len(zstd_ref.compress_with_dict(m, d, lv, False)) for m in held)
    assert ref(ours, 3) <= ref(theirs, 3) * 1.03, (ref(ours, 3), ref(theirs, 3))

    def emu(d, lv):
        trainsim.hsdict_set(d, len(d))
        buf = ctypes.create_string_buffer(8192)
        return sum(trainsim.hsdict_compress(buf, 8192, m, len(m), lv, 0, 4096) for m in held)
    for lv in (1, 2, 3):
        assert emu(ours, lv) <= emu(theirs, lv) * 1.03, lv
    trainsim.hsdict_set(None, 0)


def test_emulated_error_conditions(trainsim):
    s = log_samples(64 << 10)
    assert emu_train(trainsim, s, 255, k=200)[0] == helpers.err(70)
    assert emu_train(trainsim, s, 1000, k=1024)[0] == helpers.err(70)
    assert emu_train(trainsim, s[:4], k=200)[0] == helpers.err(72)
    assert emu_train(trainsim, s[:6])[0] == helpers.err(72)                   # 75 % of 6 leaves 4 training samples
    assert emu_train(trainsim, [b"ab"] * 3, k=200)[0] == helpers.err(72)


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CONFIGS) + ["search"])
def test_gpu_matches_the_emulation_byte_for_byte(gpu_ctx, trainsim, name):
    make, params, _ = CONFIGS[name] if name != "search" else (lambda: log_samples(3 << 20), {}, None)
    samples = make()
    r, want, k = emu_train(trainsim, samples, **params)
    assert want is not None
    got = gpu_ctx.train_dictionary(samples, CAP, **params)
    assert got == want, (name, len(got), len(want))
    assert gpu_ctx.last_train_params.k == k and gpu_ctx.last_train_params.d == params.get("d", 8)


@pytest.mark.gpu
def test_gpu_trains_a_set_larger_than_the_arena(gpu_ctx):
    samples = log_samples(256 << 20)
    got = gpu_ctx.train_dictionary(samples, CAP, k=1024)
    assert _same_selection(got, zdict_train(samples, k=1024))


@pytest.mark.gpu
def test_gpu_round_trip_and_context_unchanged(gpu_ctx, oracle):
    import zstandard_b200 as zb
    from tools import zstd_ref
    samples, held = log_samples(3 << 20), log_samples(1 << 20, base=4 << 20)[:128]
    prior = zstd_ref.train_dict(samples[:300], 16384)
    run = oracle.lib
    run.oracle_decompress_using_dict.restype = ctypes.c_uint32
    run.oracle_decompress_using_dict.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32]

    def comp(ctx):
        dsts = [np.zeros(zb.ZStdCompress.CompressBound(len(m)), dtype=np.uint8) for m in held]
        res = ctx.compress_batch_using_dict(held, dsts, level=2, checksum=True)
        return [d[:int(r)].tobytes() for d, r in zip(dsts, res)]
    try:
        gpu_ctx.load_dictionary(prior)
        before = comp(gpu_ctx)
        dic = gpu_ctx.train_dictionary(samples, CAP, k=1024)
        assert comp(gpu_ctx) == before                                       # the loaded dictionary is untouched
        gpu_ctx.load_dictionary(None)
        assert zb.train_dictionary(samples, CAP, ctx=gpu_ctx, k=1024) == dic   # also with no dictionary loaded
        gpu_ctx.load_dictionary(dic)
        frames = comp(gpu_ctx)
        outs = [np.zeros(len(m), dtype=np.uint8) for m in held]
        res = gpu_ctx.decompress_batch(frames, outs)
        for m, f, r, o in zip(held, frames, res, outs):
            assert int(r) == len(m) and o.tobytes() == m
            assert zstd_ref.decompress_with_dict(f, len(m), dic) == m
            buf = ctypes.create_string_buffer(len(m) + 8)
            assert run.oracle_decompress_using_dict(buf, len(m), f, len(f), dic, len(dic)) == len(m) and buf.raw[:len(m)] == m
    finally:
        gpu_ctx.load_dictionary(None)


@pytest.mark.gpu
def test_gpu_error_conditions(gpu_ctx):
    import zstandard_b200 as zb
    s = log_samples(64 << 10)

    def code(samples, capacity=CAP, **p):
        with pytest.raises(zb.TrainError) as e:
            gpu_ctx.train_dictionary(samples, capacity, **p)
        return e.value.code
    assert code(s, 255, k=200) == helpers.err(70)
    assert code(s, 1000, k=1024) == helpers.err(70)
    assert code(s, 1000) == helpers.err(70)                                   # the search's largest k is 1998
    assert code(s[:4], k=200) == helpers.err(72)
    assert code(s[:6]) == helpers.err(72)
    assert code([b"ab"] * 3, k=200) == helpers.err(72)
    for bad in (dict(k=200, d=7), dict(k=200, f=25), dict(k=200, accel=11), dict(k=200, level=4), dict(k=200, split_percent=101),
                dict(k=4000)):
        assert code(s, 8192, **bad) == helpers.err(1), bad
        assert gpu_ctx.last_error()
