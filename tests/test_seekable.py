"""Seekable archives (zstd's seekable format): the table writer, parser and range planner of zstandard_b200/csrc/seekable.h on a
CPU (through tests/hostsim/seekable.cpp), and on the GPU the compress and range-decode entry points against libzstd, the
oracle, compress_batch and a small Python writer and reader of the format written from its specification (the reference for
the table bytes)."""
import ctypes
import os
import random
import struct
import subprocess

import numpy as np
import pytest

from tests import helpers

SKIP_MAGIC, FOOTER_MAGIC = 0x184D2A5E, 0x8F92EAB1
E_PREFIX, E_CORRUPT, E_CHECKSUM, E_SRCSIZE = helpers.err(10), helpers.err(20), helpers.err(22), helpers.err(72)
E_DSTSMALL = helpers.err(70)


# ---- the format in Python ----------------------------------------------------------------------------------------------
def py_table(entries, ck):
    """entries: [(compressed, decompressed, checksum)] -> the table frame."""
    body = b"".join(struct.pack("<II", c, d) + (struct.pack("<I", x) if ck else b"") for c, d, x in entries)
    return struct.pack("<II", SKIP_MAGIC, len(body) + 9) + body + struct.pack("<IBI", len(entries), 0x80 if ck else 0, FOOTER_MAGIC)


def py_archive(frames, contents, ck):
    """Frames (bytes) of the given contents, then their table; checksums = low 32 bits of XXH64 of the content."""
    xs = [_xxh32(c) for c in contents] if ck else [0] * len(frames)
    return b"".join(frames) + py_table([(len(f), len(c), x) for f, c, x in zip(frames, contents, xs)], ck)


_ORACLE = None


def _xxh32(data):
    global _ORACLE
    if _ORACLE is None:
        _ORACLE = helpers.Oracle()
    return _ORACLE.xxh64(data) & 0xFFFFFFFF


def py_read(archive):
    """-> (entries, ck) or an error code (the contract of zstdb200_seekable_info_get)."""
    a = bytes(archive)
    if len(a) < 17:
        return E_SRCSIZE
    n, sfd, magic = struct.unpack("<IBI", a[-9:])
    if magic != FOOTER_MAGIC:
        return E_PREFIX
    if sfd & 0x7C:
        return E_CORRUPT
    ck = bool(sfd & 0x80)
    eb = 12 if ck else 8
    size = 8 + n * eb + 9
    if size > len(a):
        return E_SRCSIZE
    t = a[len(a) - size:]
    if struct.unpack("<I", t[:4])[0] != SKIP_MAGIC:
        return E_PREFIX
    if struct.unpack("<I", t[4:8])[0] != size - 8:
        return E_CORRUPT
    ents = []
    for i in range(n):
        e = t[8 + i * eb:8 + (i + 1) * eb]
        c, d = struct.unpack("<II", e[:8])
        ents.append((c, d, struct.unpack("<I", e[8:])[0] if ck else 0))
    if sum(c for c, _, _ in ents) != len(a) - size:
        return E_CORRUPT
    return ents, ck


def py_plan(dsizes, offset, length):
    """Brute force: [(frame, dstOff, skip, take)] of the frames that hold a byte of [offset, offset + length), or srcSize_wrong."""
    content = sum(dsizes)
    if offset + length > content:
        return E_SRCSIZE
    owner = [i for i, d in enumerate(dsizes) for _ in range(d)]
    start = np.cumsum([0] + list(dsizes))
    out = {}
    for pos in range(offset, offset + length):
        i = owner[pos]
        if i not in out:
            out[i] = [i, pos - offset, pos - int(start[i]), 0]
        out[i][3] += 1
    return [tuple(v) for _, v in sorted(out.items())]


# ---- seekable.h on the CPU ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sk():
    d = os.path.join(helpers.ROOT, "tests", "hostsim")
    path = os.path.join(d, "_build", "libseekable.so")
    deps = [os.path.join(d, "seekable.cpp"), os.path.join(helpers.ROOT, "zstandard_b200", "csrc", "seekable.h")]
    if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(x) for x in deps):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared", "-static-libstdc++", "-static-libgcc",
                        "-o", path, deps[0]], check=True)
    lib = ctypes.CDLL(path)
    p, u64 = ctypes.c_void_p, ctypes.c_uint64
    lib.sk_table_bytes.argtypes, lib.sk_table_bytes.restype = [u64, ctypes.c_int], u64
    lib.sk_write_table.argtypes = [p, ctypes.c_size_t, p, p, p, ctypes.c_int]
    lib.sk_parse.argtypes, lib.sk_parse.restype = [ctypes.c_char_p, u64, p, p], ctypes.c_uint32
    lib.sk_plan.argtypes, lib.sk_plan.restype = [ctypes.c_char_p, u64, u64, u64, p, p], ctypes.c_uint32
    return lib


def c_write(lib, entries, ck):
    n = len(entries)
    arr = np.array(entries, dtype=np.uint32).reshape(n, 3) if n else np.zeros((0, 3), dtype=np.uint32)
    cs, ds, xs = (np.ascontiguousarray(arr[:, k]) for k in range(3))
    out = np.zeros(lib.sk_table_bytes(n, int(ck)), dtype=np.uint8)
    lib.sk_write_table(out.ctypes.data, n, cs.ctypes.data, ds.ctypes.data, xs.ctypes.data, int(ck))
    return out.tobytes()


def c_parse(lib, archive):
    fields = np.zeros(7, dtype=np.uint64)
    n = len(archive) // 8 + 1
    ents = np.zeros(3 * n, dtype=np.uint32)
    r = lib.sk_parse(archive, len(archive), fields.ctypes.data, ents.ctypes.data)
    if r:
        return r
    k = int(fields[0])
    return [tuple(int(x) for x in ents[3 * i:3 * i + 3]) for i in range(k)], bool(fields[1]), [int(x) for x in fields]


def c_plan(lib, archive, offset, length, nmax):
    out = np.zeros(6 * (nmax + 1), dtype=np.uint64)
    cnt = np.zeros(1, dtype=np.uint64)
    r = lib.sk_plan(archive, len(archive), offset, length, out.ctypes.data, cnt.ctypes.data)
    return r, [tuple(int(x) for x in out[6 * k:6 * k + 6]) for k in range(int(cnt[0]))]


@pytest.mark.parametrize("n", [0, 1, 3, 70000])
@pytest.mark.parametrize("ck", [False, True])
def test_table_round_trip(sk, n, ck):
    rng = random.Random(n * 2 + ck)
    ents = [(rng.randrange(1, 1 << 20 if n < 100 else 40), rng.randrange(0, 1 << 32), rng.randrange(1 << 32) if ck else 0) for _ in range(n)]
    t = py_table(ents, ck)
    assert c_write(sk, ents, ck) == t
    archive = bytes(sum(c for c, _, _ in ents)) + t   # a data section of the right length in front of the table
    got = c_parse(sk, archive)
    assert got[0] == ents and got[1] == ck and py_read(archive) == (ents, ck)
    f = got[2]
    assert f[2] == len(t) and f[3] == len(archive) - len(t) and f[4] == sum(d for _, d, _ in ents)
    assert f[5] == max([d for _, d, _ in ents], default=0) and f[6] == max([c for c, _, _ in ents], default=0)


def test_frame_size_field_limits_the_frame_count(sk):
    sk.sk_table_fits.argtypes, sk.sk_table_fits.restype = [ctypes.c_uint64, ctypes.c_int], ctypes.c_int
    for ck, eb in ((True, 12), (False, 8)):
        top = (0xFFFFFFFF - 9) // eb
        assert top * eb + 9 <= 0xFFFFFFFF < (top + 1) * eb + 9
        assert sk.sk_table_fits(top, int(ck)) == 1 and sk.sk_table_fits(top + 1, int(ck)) == 0
    assert sk.sk_table_fits(0, 1) == 1


def _malformed():
    ents = [(5, 7, 0x11111111), (3, 0, 0x22222222), (4, 9, 0x33333333)]
    good = b"\1" * 12 + py_table(ents, True)
    cases = {"ok": (good, 0)}
    b = bytearray(good); b[-1] ^= 0xFF
    cases["footer magic"] = (bytes(b), E_PREFIX)
    for bit in range(2, 7):
        b = bytearray(good); b[-5] |= 1 << bit
        cases[f"reserved bit {bit}"] = (bytes(b), E_CORRUPT)
    for bit in (0, 1):
        b = bytearray(good); b[-5] |= 1 << bit
        cases[f"ignored bit {bit}"] = (bytes(b), 0)
    b = bytearray(good); b[12] ^= 1
    cases["skippable magic"] = (bytes(b), E_PREFIX)
    b = bytearray(good); b[16] += 1
    cases["frame size"] = (bytes(b), E_CORRUPT)
    b = bytearray(good); b[-9] = 200
    cases["table longer than archive"] = (bytes(b), E_SRCSIZE)
    cases["sizes short of the data"] = (b"\1" + good, E_CORRUPT)
    cases["sizes past the data"] = (good[1:], E_CORRUPT)
    b = bytearray(good); b[20] += 1
    cases["sizes past the data, table intact"] = (bytes(b), E_CORRUPT)
    for k in range(17):
        cases[f"{k} bytes"] = (good[len(good) - k:], E_SRCSIZE)
    cases["17-byte empty archive"] = (py_table([], False), 0)
    return cases


@pytest.mark.parametrize("name", list(_malformed()))
def test_malformed_tables(sk, name):
    archive, want = _malformed()[name]
    got = c_parse(sk, archive)
    py = py_read(archive)
    if want:
        assert got == want and py == want
    else:
        assert isinstance(got, tuple) and got[:2] == py


@pytest.mark.parametrize("dsizes", [[3, 1, 4, 0, 1, 5], [7], [0, 2, 0, 0, 3, 0], [1, 1, 1]])
def test_range_plan_exhaustive(sk, dsizes):
    csizes = [10 + i for i in range(len(dsizes))]
    archive = b"".join(bytes([i]) * c for i, c in enumerate(csizes)) + py_table([(c, d, 0) for c, d in zip(csizes, dsizes)], False)
    content = sum(dsizes)
    src_off = np.cumsum([0] + csizes)
    for off in range(content + 2):
        for ln in range(content + 2 - off):
            r, got = c_plan(sk, archive, off, ln, len(dsizes))
            want = py_plan(dsizes, off, ln)
            if want == E_SRCSIZE:
                assert r == E_SRCSIZE and got == [], (off, ln)
                continue
            assert r == 0
            assert [g[:4] for g in got] == want, (off, ln)
            assert all(dsizes[g[0]] > 0 and g[4] == src_off[g[0]] and g[5] == csizes[g[0]] for g in got)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
FS = 4096
LEVELS = [1, 2, 3, -1, -7]


def _data(n, seed=5):
    from tools import corpus
    return corpus.log(n, (seed, 24)).tobytes()


def split_archive(archive):
    ents, ck = py_read(archive)
    frames, pos = [], 0
    for c, _, _ in ents:
        frames.append(archive[pos:pos + c])
        pos += c
    return frames, ents, ck


def check_archive(ctx, oracle, data, fs, level, checksum, archive):
    from tools import zstd_ref
    got = py_read(archive)
    assert isinstance(got, tuple), got
    frames, ents, ck = split_archive(archive)
    chunks = [data[i:i + fs] for i in range(0, len(data), fs)]
    assert ck == bool(checksum) and len(frames) == len(chunks)
    if chunks:
        import zstandard_b200 as zb
        outs = [np.zeros(zb.ZStdCompress.CompressBound(len(c)), dtype=np.uint8) for c in chunks]
        res = ctx.compress_batch(chunks, outs, level=level, checksum=checksum)
        for k, (f, o, r, c, e) in enumerate(zip(frames, outs, res, chunks, ents)):
            assert f == o[:int(r)].tobytes(), k
            assert e[0] == len(f) and e[1] == len(c)
            if checksum:
                assert e[2] == struct.unpack("<I", f[-4:])[0] == _xxh32(c)
            ro, oo, _ = oracle.decompress(f, len(c))
            assert ro == len(c) and oo == c, k
    assert (zstd_ref.decompress(archive, len(data)) or b"") == data


def _sizes(fs):
    return [0, 1, fs - 1, fs, 7 * fs, 7 * fs + 1]


@pytest.mark.gpu
@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("checksum", [False, True])
def test_compress_seekable(gpu_ctx, oracle, level, checksum):
    for size in _sizes(FS):
        data = _data(size, 11 + size)
        archive = gpu_ctx.compress_seekable(data, FS, level=level, checksum=checksum)
        check_archive(gpu_ctx, oracle, data, FS, level, checksum, archive)
    assert len(gpu_ctx.compress_seekable(b"", FS, level=level, checksum=checksum)) == 17


@pytest.fixture(scope="module")
def small_ctx():
    import zstandard_b200 as zb
    ctx = zb.Context(max_batch_bytes=1 << 20)
    yield ctx
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("checksum", [False, True])
def test_compress_seekable_more_frames_and_bytes_than_one_batch(small_ctx, oracle, level, checksum):
    fs = 17
    n = small_ctx.max_items + 500
    data = _data(n * fs - 3, 7)
    assert len(data) > small_ctx.max_batch_bytes and n > small_ctx.max_items
    archive = small_ctx.compress_seekable(data, fs, level=level, checksum=checksum)
    check_archive(small_ctx, oracle, data, fs, level, checksum, archive)


def _torch_u8(b, slack=8):
    import torch
    t = torch.zeros(len(b) + slack, dtype=torch.uint8, device="cuda:0")
    if b:
        t[:len(b)] = torch.frombuffer(bytearray(b), dtype=torch.uint8).to("cuda:0")
    return t


def device_compress(ctx, data, fs, level, checksum):
    import torch
    src = _torch_u8(data)
    cap = ctx.seekable_bound(len(data), fs)
    dst = torch.zeros(cap + 64, dtype=torch.uint8, device="cuda:0")
    dst[cap:] = 0xA5
    size = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    ctx.compress_seekable_device(level, checksum, fs, src.data_ptr(), len(data), dst.data_ptr(), cap, size.data_ptr())
    torch.cuda.synchronize()
    n = int(size.item())
    assert (dst[cap:] == 0xA5).all()
    return dst[:n].cpu().numpy().tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("checksum", [False, True])
def test_device_compress_matches_host(gpu_ctx, level, checksum):
    for size in _sizes(FS) + [300 * FS + 5]:
        data = _data(size, 3 + size)
        assert device_compress(gpu_ctx, data, FS, level, checksum) == gpu_ctx.compress_seekable(data, FS, level=level, checksum=checksum)


def _archives():
    """(name, content, archive): the project's own, and the Python writer's around libzstd frames with and without frame and
    table checksums (frames of uneven sizes, one of no content)."""
    import zstandard_b200 as zb  # noqa: F401
    from tools import zstd_ref
    rng = random.Random(9)
    out = []
    data = _data(37 * 3000 + 77, 21)
    sizes = [rng.choice([1, 100, 3000, 4096, 9000]) for _ in range(40)] + [0, 5]
    content = _data(sum(sizes), 22)
    pos, chunks = 0, []
    for s in sizes:
        chunks.append(content[pos:pos + s])
        pos += s
    for fck in (False, True):
        for tck in (False, True):
            frames = [zstd_ref.compress(c, level=3, checksum=fck) for c in chunks]
            out.append((f"libzstd frame_ck={fck} table_ck={tck}", content, py_archive(frames, chunks, tck)))
    return data, out


def _ranges(content_len, rng):
    L = content_len
    rs = [(0, L), (0, 0), (L // 2, 0), (10, 100), (2990, 20), (1000, L // 2), (L - 1234, 1234), (L - 1, 1)]
    for _ in range(200):
        a = rng.randrange(L + 1)
        rs.append((a, rng.randrange(L - a + 1)))
    return rs


def host_decode(ctx, archive, off, ln, guard=64):
    buf = np.full(ln + 2 * guard, 0xA5, dtype=np.uint8)
    out = buf[guard:guard + ln]
    import zstandard_b200 as zb
    try:
        ctx.decompress_seekable(archive, off, ln, out=out)
        code = 0
    except zb.SeekableError as e:
        code = e.code
    assert (buf[:guard] == 0xA5).all() and (buf[guard + ln:] == 0xA5).all()
    return code, out.tobytes()


def device_decode(ctx, archive, off, ln, guard=64, t_src=None):
    import torch
    src = t_src if t_src is not None else _torch_u8(archive, 0)
    buf = torch.full((ln + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda:0")
    code = torch.full((1,), 7, dtype=torch.int32, device="cuda:0")
    ctx.decompress_seekable_device(buf.data_ptr() + guard, off, ln, src.data_ptr(), len(archive), code.data_ptr())
    torch.cuda.synchronize()
    b = buf.cpu().numpy()
    assert (b[:guard] == 0xA5).all() and (b[guard + ln:] == 0xA5).all()
    return int(code.item()) & 0xFFFFFFFF, b[guard:guard + ln].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["host", "device"])
def test_range_decode(gpu_ctx, variant):
    data, archives = _archives()
    archives = [("own level 3 ck", data, gpu_ctx.compress_seekable(data, 3000, 3, True)),
                ("own level -1", data, gpu_ctx.compress_seekable(data, 3000, -1, False))] + archives
    rng = random.Random(1 if variant == "host" else 2)
    for name, content, archive in archives:
        t_src = _torch_u8(archive, 0) if variant == "device" else None
        for off, ln in _ranges(len(content), rng):
            if variant == "host":
                code, got = host_decode(gpu_ctx, archive, off, ln)
            else:
                code, got = device_decode(gpu_ctx, archive, off, ln, t_src=t_src)
            assert code == 0 and got == content[off:off + ln], (name, off, ln, hex(code))


def _decode(ctx, variant, archive, off, ln):
    return host_decode(ctx, archive, off, ln) if variant == "host" else device_decode(ctx, archive, off, ln)


def _set_entry(archive, i, field, value):
    ents, ck = py_read(archive)
    eb = 12 if ck else 8
    tpos = len(archive) - (8 + len(ents) * eb + 9)
    b = bytearray(archive)
    struct.pack_into("<I", b, tpos + 8 + i * eb + 4 * field, value)
    return bytes(b)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["host", "device"])
def test_range_decode_errors(gpu_ctx, oracle, variant):
    from tools import zstd_ref
    data = _data(20 * 3000, 31)
    own = gpu_ctx.compress_seekable(data, 3000, 3, True)
    L = len(data)
    # a range past the end: srcSize_wrong and nothing written (the guards cover the whole destination)
    for off, ln in ((0, L + 1), (L, 1), (L + 5, 0)):
        code, got = _decode(gpu_ctx, variant, own, off, ln)
        assert code == E_SRCSIZE and got == b"\xa5" * ln
    # a table error reaches the code too
    b = bytearray(own); b[-1] ^= 1
    assert _decode(gpu_ctx, variant, bytes(b), 0, 10)[0] == E_PREFIX
    assert _decode(gpu_ctx, variant, b"\0" * 5, 0, 0)[0] == E_SRCSIZE
    # a wrong table checksum, for frames with their own checksum and for frames without one
    ents, _ = py_read(own)
    bad = _set_entry(own, 7, 2, ents[7][2] ^ 1)
    assert _decode(gpu_ctx, variant, bad, 0, L)[0] == E_CHECKSUM
    assert _decode(gpu_ctx, variant, bad, 0, 7 * 3000)[0] == 0        # frame 7 is not in this range
    chunks = [data[i:i + 3000] for i in range(0, L, 3000)]
    plain = py_archive([zstd_ref.compress(c, 3, checksum=False) for c in chunks], chunks, True)
    ents, _ = py_read(plain)
    bad = _set_entry(plain, 4, 2, ents[4][2] ^ 0x80000000)
    assert _decode(gpu_ctx, variant, bad, 100, L - 200)[0] == E_CHECKSUM
    # the first error in archive order wins
    two = _set_entry(_set_entry(plain, 9, 2, ents[9][2] ^ 1), 6, 1, ents[6][1] + 1)
    assert _decode(gpu_ctx, variant, two, 0, L)[0] == E_CORRUPT
    # an entry that lies about its decompressed size, either way
    for delta in (1, -1):
        lied = _set_entry(plain, 3, 1, ents[3][1] + delta)
        assert _decode(gpu_ctx, variant, lied, 0, L + delta)[0] == E_CORRUPT
    # a corrupted frame: the code the oracle gives that frame (a capacity of the entry's size that is too small, or a content of
    # another size, is the entry's corruption_detected)
    frames, ents, _ = split_archive(own)
    rng = random.Random(4)
    for trial in range(12):
        k = rng.randrange(len(frames))
        f = bytearray(frames[k])
        for _ in range(3):
            f[rng.randrange(6, len(f))] ^= 1 << rng.randrange(8)
        fr = frames[:k] + [bytes(f)] + frames[k + 1:]
        arch = b"".join(fr) + py_table(ents, True)
        ro, oo, _ = oracle.decompress(bytes(f), ents[k][1])
        want = ro
        if ro == E_DSTSMALL or (not helpers.is_err(ro) and ro != ents[k][1]):
            want = E_CORRUPT
        elif not helpers.is_err(ro) and _xxh32(oo) != ents[k][2]:
            want = E_CHECKSUM
        assert _decode(gpu_ctx, variant, arch, 0, L)[0] == want, (trial, k, hex(ro))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["host", "device"])
def test_frame_larger_than_the_context_fails_the_call(small_ctx, variant):
    from tools import zstd_ref
    big = _data(3 << 20, 41)
    arch = py_archive([zstd_ref.compress(big, 1, checksum=False), zstd_ref.compress(b"abc", 1)], [big, b"abc"], False)
    with pytest.raises(RuntimeError, match="larger than the context"):
        _decode(small_ctx, variant, arch, 0, len(big) + 3)
    # a range that only needs the small frame works
    assert _decode(small_ctx, variant, arch, len(big) + 1, 2) == (0, b"bc")


# The constant: one k_seek_check per slice on the host path (one slice here) and per group on the device path.  A device range
# that cuts its first and last frame is two groups: those two frames decode into scratch in one launch sequence of their own
# (the decode pipeline writes every item of a launch through one destination base), then the rest straight into dst.
SEEK_CHECK_LAUNCHES = 1


@pytest.mark.gpu
def test_one_batch_not_a_pass_per_frame(gpu_ctx):
    n, fs = 512, 4096
    data = _data(n * fs, 51)
    archive = gpu_ctx.compress_seekable(data, fs, 3, True)
    frames, _, _ = split_archive(archive)
    l0 = gpu_ctx.kernel_launches
    outs = [np.zeros(fs, dtype=np.uint8) for _ in frames]
    assert (gpu_ctx.decompress_batch(frames, outs) == fs).all()
    base = gpu_ctx.kernel_launches - l0
    l0 = gpu_ctx.kernel_launches
    assert host_decode(gpu_ctx, archive, 100, n * fs - 200) == (0, data[100:n * fs - 100])
    assert gpu_ctx.kernel_launches - l0 <= base + SEEK_CHECK_LAUNCHES
    l0 = gpu_ctx.kernel_launches
    assert device_decode(gpu_ctx, archive, 0, n * fs) == (0, data)
    assert gpu_ctx.kernel_launches - l0 <= base + SEEK_CHECK_LAUNCHES
    # the launch sequence of the two edge frames alone
    l0 = gpu_ctx.kernel_launches
    assert (gpu_ctx.decompress_batch([frames[0], frames[-1]], [np.zeros(fs, dtype=np.uint8) for _ in range(2)]) == fs).all()
    edge = gpu_ctx.kernel_launches - l0
    l0 = gpu_ctx.kernel_launches
    assert device_decode(gpu_ctx, archive, 100, n * fs - 200) == (0, data[100:n * fs - 100])
    assert gpu_ctx.kernel_launches - l0 <= base + edge + 2 * SEEK_CHECK_LAUNCHES


@pytest.mark.gpu
def test_one_context_over_two_devices_seekable(gpu_ctx):
    import torch
    import zstandard_b200 as zb
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ctx2 = zb.Context(devices=[0, 1], max_batch_bytes=4 << 20)
    try:
        data = _data(9 << 20, 61)
        a1 = gpu_ctx.compress_seekable(data, 65536, 3, True)
        a2 = ctx2.compress_seekable(data, 65536, 3, True)
        assert a1 == a2
        rng = random.Random(5)
        for off, ln in [(0, len(data))] + [(a, rng.randrange(len(data) - a + 1)) for a in (rng.randrange(len(data)) for _ in range(20))]:
            assert host_decode(ctx2, a2, off, ln) == host_decode(gpu_ctx, a1, off, ln) == (0, data[off:off + ln])
    finally:
        ctx2.close()


@pytest.mark.gpu
def test_existing_decoder_reads_an_archive_as_one_item(gpu_ctx):
    data = _data(8 * 5000 - 17, 71)
    for ck in (False, True):
        archive = gpu_ctx.compress_seekable(data, 5000, 2, ck)
        out = np.zeros(len(data), dtype=np.uint8)
        res = gpu_ctx.decompress_batch([archive], [out])
        assert int(res[0]) == len(data) and out.tobytes() == data
        info = gpu_ctx.seekable_info(archive)
        assert (info.n_frames, info.content_size, info.checksums, info.max_frame_content) == (8, len(data), int(ck), 5000)
        assert info.data_size == len(archive) - (8 + 8 * (12 if ck else 8) + 9)


@pytest.mark.gpu
def test_too_many_frames_for_the_table_fail_before_any_work(gpu_ctx):
    import zstandard_b200 as zb
    lib = zb.load_library()
    n = (0xFFFFFFFF - 9) // 12 + 1                 # one frame more than Frame_Size holds with checksums
    src = np.zeros(n, dtype=np.uint8)
    dst = np.zeros(64, dtype=np.uint8)
    size = ctypes.c_uint64(0)
    for ck, why in ((1, "Frame_Size"), (0, "seekable_bound")):   # without checksums the count fits: the capacity check speaks
        rc = lib.zstdb200_compress_seekable(gpu_ctx.handle, 1, ck, 1, src.ctypes.data, n, dst.ctypes.data, dst.size, ctypes.byref(size))
        assert rc != 0 and why in gpu_ctx.last_error(), gpu_ctx.last_error()


def _entry_archive(parts, contents):
    """Python-written archive whose entry i is the bytes parts[i] (one or more frames) of content contents[i], table checksums on."""
    return b"".join(parts) + py_table([(len(p), len(c), _xxh32(c)) for p, c in zip(parts, contents)], True)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["host", "device"])
def test_entry_spans_beyond_the_frame(gpu_ctx, variant):
    from tools import zstd_ref
    a, b = _data(5000, 81), _data(3000, 82)
    fa, fb = zstd_ref.compress(a, 3, checksum=True), zstd_ref.compress(b, 3, checksum=True)
    skip = struct.pack("<II", 0x184D2A50, 6) + b"padpad"
    # a skippable frame after a checksummed frame inside its entry: the table checksum is compared with the verified trailer
    ok = _entry_archive([fa + skip, fb], [a, b])
    assert _decode(gpu_ctx, variant, ok, 0, 8000) == (0, a + b)
    # and a wrong table checksum is still caught there
    ents, _ = py_read(ok)
    assert _decode(gpu_ctx, variant, _set_entry(ok, 0, 2, ents[0][2] ^ 1), 0, 8000)[0] == E_CHECKSUM
    # an entry that holds two data frames is not one frame
    two = _entry_archive([fa + fb], [a + b])
    assert _decode(gpu_ctx, variant, two, 0, 8000)[0] == E_CORRUPT


@pytest.mark.gpu
def test_calls_right_after_a_device_range_decode_do_not_disturb_it(gpu_ctx):
    """decompress_seekable_device returns with its uploads and kernels queued on the caller's stream.  Host and device calls
    made at once after it, with no synchronisation, must neither change what it decodes nor be changed by it."""
    import torch
    n, fs = 600, 4096
    data = _data(n * fs, 91)
    archive = gpu_ctx.compress_seekable(data, fs, 1, True)
    other = _data(40 * fs, 92)
    other_arc = gpu_ctx.compress_seekable(other, fs, 3, False)
    t_src = _torch_u8(archive, 0)
    st = torch.cuda.Stream()
    for off, ln in ((0, n * fs), (777, n * fs - 2000)):
        out = torch.full((ln,), 0xA5, dtype=torch.uint8, device="cuda:0")
        code = torch.full((1,), 7, dtype=torch.int32, device="cuda:0")
        with torch.cuda.stream(st):
            torch.cuda._sleep(50_000_000)          # keeps the call's queued work waiting behind a kernel on its stream
        gpu_ctx.decompress_seekable_device(out.data_ptr(), off, ln, t_src.data_ptr(), len(archive), code.data_ptr(),
                                           stream=st.cuda_stream)
        # at once, no synchronisation: a host batch call, a host seekable call and a device call on another stream
        frames, _, _ = split_archive(other_arc)
        outs = [np.zeros(fs, dtype=np.uint8) for _ in frames]
        assert (gpu_ctx.decompress_batch(frames, outs) == fs).all() and b"".join(o.tobytes() for o in outs) == other
        assert gpu_ctx.decompress_seekable(other_arc, 5, 30000) == other[5:30005]
        assert device_compress(gpu_ctx, other, fs, 3, False) == other_arc
        torch.cuda.synchronize()
        assert int(code.item()) == 0 and out.cpu().numpy().tobytes() == data[off:off + ln]
