"""The host path's batch plan (zstandard_b200/csrc/host_plan.h) on a CPU, through a g++ build of tests/hostsim/host_plan.cpp:
sub-batches that fit the device arenas, the re-cut that gives every device of a context a share, the slices dealt to the
streams, the descriptor layout, and the test that lets back-to-back caller buffers skip the staging."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from tests import helpers

MiB = 1 << 20


@pytest.fixture(scope="module")
def plan():
    d = os.path.join(helpers.ROOT, "tests", "hostsim")
    path = os.path.join(d, "_build", "libhost_plan.so")
    deps = [os.path.join(d, "host_plan.cpp"), os.path.join(helpers.ROOT, "zstandard_b200", "csrc", "host_plan.h")]
    if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(x) for x in deps):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared", "-static-libstdc++", "-static-libgcc",
                        "-o", path, deps[0]], check=True)
    lib = ctypes.CDLL(path)
    sz, p = ctypes.c_size_t, ctypes.c_void_p
    lib.hp_subbatches.argtypes = [sz, sz, sz, sz, p, p, p, ctypes.POINTER(ctypes.c_int)]
    lib.hp_split.argtypes = [p, sz, sz, p, p, p]
    lib.hp_slices.argtypes = [p, p, sz, ctypes.c_int, sz, p]
    lib.hp_back_to_back.argtypes = [p, p, sz, sz, sz]
    lib.hp_desc_layout.argtypes = [sz, p]
    lib.hp_min_slice_items.argtypes = [ctypes.c_int]
    for f in (lib.hp_subbatches, lib.hp_split, lib.hp_slices, lib.hp_min_slice_items):
        f.restype = sz
    return lib


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def _ranges(out, k):
    return [(int(out[2 * i]), int(out[2 * i + 1])) for i in range(k)]


def subbatches(lib, ins, outs, max_in, max_out, max_items):
    ins, outs = _u32(ins), _u32(outs)
    n = len(ins)
    out = np.zeros(2 * max(n, 1), dtype=np.uint64)
    big = ctypes.c_int(0)
    k = lib.hp_subbatches(n, max_in, max_out, max_items,
                          ins.ctypes.data, outs.ctypes.data, out.ctypes.data, ctypes.byref(big))
    return _ranges(out, k), bool(big.value)


def split(lib, subs, nd, ins, outs):
    ins, outs = _u32(ins), _u32(outs)
    r = np.array(subs, dtype=np.uint64).reshape(-1)
    out = np.zeros(2 * (len(ins) + len(subs) * nd + 1), dtype=np.uint64)
    k = lib.hp_split(r.ctypes.data, len(subs), nd, ins.ctypes.data, outs.ctypes.data, out.ctypes.data)
    return _ranges(out, k)


def slices(lib, src, cap, decode, slice_bytes=32 * MiB):
    src, cap = _u32(src), _u32(cap)
    out = np.zeros(2 * max(len(src), 1), dtype=np.uint64)
    k = lib.hp_slices(src.ctypes.data, cap.ctypes.data, len(src), int(decode), slice_bytes,
                      out.ctypes.data)
    return _ranges(out, k)


def back_to_back(lib, addrs, sizes, slack, limit):
    a = np.array(addrs, dtype=np.uint64)
    s = _u32(sizes)
    return bool(lib.hp_back_to_back(a.ctypes.data, s.ctypes.data, len(s), slack, limit))


def a16(v):
    return (int(v) + 15) // 16 * 16


def assert_partition(ranges, n):
    """consecutive, non-empty, in order, covering [0, n) exactly once"""
    assert ranges and ranges[0][0] == 0 and ranges[-1][1] == n
    for (lo, hi), (lo2, _) in zip(ranges, ranges[1:]):
        assert lo < hi == lo2
    assert ranges[-1][0] < ranges[-1][1]


def test_every_item_in_one_subbatch_and_one_slice_within_the_arena_limits(plan):
    rng = random.Random(1)
    for trial in range(40):
        n = rng.randint(1, 3000)
        ins = [rng.choice([0, 1, 17, 4096, 65536, 200000, rng.randrange(1 << 20)]) for _ in range(n)]
        outs = [rng.choice([0, 5, 4096, 131072, rng.randrange(1 << 20)]) for _ in range(n)]
        max_in, max_out = rng.choice([2, 8, 64]) * MiB, rng.choice([2, 8, 64]) * MiB
        max_items = rng.choice([16, 1000, 65536])
        subs, big = subbatches(plan, ins, outs, max_in, max_out, max_items)
        assert not big
        assert_partition(subs, n)
        for lo, hi in subs:
            assert hi - lo <= max_items
            assert sum(a16(x) for x in ins[lo:hi]) <= max_in and sum(a16(x) for x in outs[lo:hi]) <= max_out
            if hi < n and hi - lo < max_items:   # greedy: the next item did not fit
                assert (sum(a16(x) for x in ins[lo:hi + 1]) > max_in) or (sum(a16(x) for x in outs[lo:hi + 1]) > max_out)
            for decode in (0, 1):
                sl = slices(plan, ins[lo:hi], outs[lo:hi], decode, rng.choice([1, 32]) * MiB)
                assert_partition(sl, hi - lo)


def test_a_lone_item_larger_than_the_arena_is_reported(plan):
    _, big = subbatches(plan, [10, 2 * MiB + 1, 10], [10, 10, 10], 2 * MiB, 2 * MiB, 100)
    assert big
    _, big = subbatches(plan, [10, 10], [10, 2 * MiB - 15], 2 * MiB, 2 * MiB - 8, 100)   # 16-byte alignment pushes it over
    assert big
    subs, big = subbatches(plan, [10, 10], [10, 2 * MiB - 24], 2 * MiB, 2 * MiB - 8, 100)
    assert not big and subs == [(0, 1), (1, 2)]


def test_hand_computed_subbatches_and_device_shares(plan):
    # aligned inputs 16, 32, 32, 16 against 64 bytes: 16 + 32, then 32 + 16
    assert subbatches(plan, [10, 20, 30, 5], [0, 0, 0, 0], 64, 1000, 100) == ([(0, 2), (2, 4)], False)
    assert subbatches(plan, [1] * 5, [1] * 5, 1000, 1000, 2) == ([(0, 2), (2, 4), (4, 5)], False)
    assert subbatches(plan, [], [], 1000, 1000, 2) == ([], False)
    # costs in + out + 1
    assert split(plan, [(0, 4)], 2, [10] * 4, [0] * 4) == [(0, 2), (2, 4)]
    assert split(plan, [(0, 4)], 2, [99, 0, 0, 0], [0] * 4) == [(0, 1), (1, 4)]
    assert split(plan, [(0, 4)], 2, [0, 0, 0, 99], [0] * 4) == [(0, 3), (3, 4)]
    assert split(plan, [(0, 3)], 4, [5] * 3, [5] * 3) == [(0, 1), (1, 2), (2, 3)]
    assert split(plan, [(0, 1)], 8, [5], [5]) == [(0, 1)]
    assert split(plan, [(0, 2), (2, 5)], 1, [1] * 5, [1] * 5) == [(0, 2), (2, 5)]   # one device: unchanged
    assert split(plan, [(0, 2), (2, 5)], 2, [1] * 5, [1] * 5) == [(0, 2), (2, 5)]   # as many sub-batches as devices
    assert split(plan, [(0, 2), (2, 5)], 3, [1] * 5, [1] * 5) == [(0, 1), (1, 2), (2, 3), (3, 4), (4, 5)]


def test_multi_device_cut_gives_every_device_a_balanced_share(plan):
    rng = random.Random(2)
    for trial in range(60):
        nd = rng.choice([2, 3, 4, 8])
        n = rng.randint(nd, 400)
        ins = [rng.choice([0, 100, 4096, 65536, rng.randrange(1 << 20)]) for _ in range(n)]
        outs = [rng.choice([0, 4096, 131072, rng.randrange(1 << 20)]) for _ in range(n)]
        cut = split(plan, [(0, n)], nd, ins, outs)
        assert len(cut) == nd
        assert_partition(cut, n)
        cost = [i + o + 1 for i, o in zip(ins, outs)]
        total, biggest = sum(cost), max(cost)
        for lo, hi in cut:
            # each share ends within one item of its byte-proportional boundary
            assert abs(sum(cost[lo:hi]) - total / nd) <= 2 * biggest


def test_decode_slices_shrink_four_two_one_and_encode_slices_do_not(plan):
    dmin, emin = plan.hp_min_slice_items(1), plan.hp_min_slice_items(0)
    assert (dmin, emin) == (1024, 512)
    # few large items: the item minimum decides (decode: a quarter for two slices, a half for two more)
    n = 4000
    sl = slices(plan, [MiB] * n, [MiB] * n, True)
    assert [hi - lo for lo, hi in sl[:6]] == [256, 256, 512, 512, 1024, 1024]
    sl = slices(plan, [MiB] * n, [MiB] * n, False)
    assert all(hi - lo == 512 for lo, hi in sl[:-1])
    # many small items: the byte target decides, shrunk the same way (4 KiB items, 32 MiB slices)
    n = 40000
    sl = slices(plan, [4096] * n, [4096] * n, True)
    assert [hi - lo for lo, hi in sl[:6]] == [2048, 2048, 4096, 4096, 8192, 8192]
    sl = slices(plan, [100] * n, [4096] * n, False)
    assert [hi - lo for lo, hi in sl] == [8192] * 4 + [n - 4 * 8192]
    # the larger of source and capacity counts; a small call is one slice
    assert slices(plan, [4096] * 10, [0] * 10, True) == [(0, 10)]
    assert slices(plan, [5], [7], False) == [(0, 1)]


def test_descriptor_layout_and_back_to_back_buffers(plan):
    out = np.zeros(5, dtype=np.uint64)
    plan.hp_desc_layout(3, out.ctypes.data)
    assert list(out) == [0, 24, 48, 60, 72]
    base = 1 << 20
    # sources: each starts where the previous ends or up to 64 bytes later, inside the limit
    assert back_to_back(plan, [base, base + 10, base + 30], [10, 20, 5], 64, 1 << 30)
    assert back_to_back(plan, [base, base + 10 + 64], [10, 20], 64, 1 << 30)
    assert not back_to_back(plan, [base, base + 10 + 65], [10, 20], 64, 1 << 30)
    assert not back_to_back(plan, [base, base + 9], [10, 20], 64, 1 << 30)           # overlap
    assert not back_to_back(plan, [base + 100, base], [10, 20], 64, 1 << 30)         # out of order
    # destinations: exactly adjacent
    assert back_to_back(plan, [base, base + 10], [10, 20], 0, 1 << 30)
    assert not back_to_back(plan, [base, base + 11], [10, 20], 0, 1 << 30)
    # the span from the first start to the last end must fit the limit
    assert back_to_back(plan, [base, base + 10], [10, 20], 0, 30)
    assert not back_to_back(plan, [base, base + 10], [10, 20], 0, 29)
    assert back_to_back(plan, [base], [0], 0, 0)
    assert not back_to_back(plan, [0, 10], [10, 20], 64, 1 << 30)                     # null first buffer
