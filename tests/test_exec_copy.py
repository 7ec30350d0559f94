"""The execute stage's flattened copies (zstandard_b200/csrc/zb_exec_copy.cuh) on seeded sets of runs, byte for byte.

k_exec and k_exec_big move the short literal runs, RLE fills and non-overlapping matches of a group of 32 sequences with the
whole warp at once, in 4-byte units that the lanes share out.  Neighbouring runs share destination words,
so a store that writes one byte too many corrupts another run's output, a match of a later round or the next frame, and only
some alignments expose it.  The frame-level suites reach the alignments their corpora happen to produce; here every case is
built to a plan:

- run lengths 0..127, all 8 destination and all 8 source alignments (of an 8-byte word);
- runs packed back to back (gap 0) or with unowned bytes between them, and lanes without a run;
- matches with off == ml, off just above ml, and sources that end exactly at the group's first byte.

tests/gpu_harness/exec_copy.cu runs one warp per case; every byte of the buffer is compared with a serial NumPy copy of the
runs, so no byte outside a run (a sentinel before, between or after the runs) may change.  On the CPU the cases' reference is
held to a byte-serial memmove model, and the harness is compiled for sm_100a."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from tests import helpers

CSRC = os.path.join(helpers.ROOT, "zstandard_b200", "csrc")
HIST = 256                    # bytes before each group a match may read
SPAN = 32 * 160               # room for 32 runs of up to 127 bytes and their gaps
LIT_ROOM = 32 * 128 + 64
KINDS = ("literals", "rle", "matches")


def _stale(path, deps):
    return not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(d) for d in deps)


def build_harness():
    """nvcc build of tests/gpu_harness/exec_copy.cu with the product's flags (sm_100a, static cudart)."""
    from zstandard_b200 import build as zbuild
    d = os.path.join(helpers.ROOT, "tests", "gpu_harness")
    path = os.path.join(d, "_build", "libexec_copy.so")
    src = os.path.join(d, "exec_copy.cu")
    deps = [src] + [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cuh", ".h"))]
    if _stale(path, deps):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        subprocess.run([nvcc] + zbuild.NVCC_FLAGS + ["-shared", "-o", path, src], check=True)
    lib = ctypes.CDLL(path)
    vp = ctypes.c_void_p
    lib.exec_copy_run.argtypes = [ctypes.c_uint32, vp, vp, vp, ctypes.c_uint64, vp, ctypes.c_uint64]
    lib.exec_copy_run.restype = ctypes.c_int
    return lib


# ---------------------------------------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------------------------------------
def _length(rng):
    r = rng.random()
    if r < 0.1:
        return 0
    if r < 0.6:
        return rng.randint(1, 16)
    if r < 0.85:
        return rng.randint(17, 40)
    return rng.randint(41, 127)


def make_case(rng, kind, g_align, src_align, sparse=False):
    """One group: its runs (dpos, spos or off, len) for 32 lanes, g's alignment in the buffer, the literal base's alignment.
    A sparse group has 1-4 short runs on random lanes: few enough units for the copies' one-row passes (U = 1)."""
    runs, pos = [], 0
    dense = rng.random() < 0.5                                  # packed back to back: neighbouring runs share words
    lanes = set(rng.sample(range(32), rng.randint(1, 4))) if sparse else set(range(32))
    for lane in range(32):
        n = rng.randint(1, 24) if sparse else _length(rng)
        if lane not in lanes or n == 0 or rng.random() < 0.05:
            runs.append([pos, 0, 0])                                # an empty lane
            continue
        if not dense:
            pos += rng.choice((0, 0, 1, 2, 3, 5, 7, 8, 9, 13))
        runs.append([pos, 0, n])
        pos += n
    if kind == "literals":
        lpos = 0
        for r in runs:                                          # literal sources in order, every source alignment
            if r[2]:
                lpos += rng.choice((0, 0, 0, 1, 3))
                r[1] = lpos
                lpos += r[2]
    elif kind == "matches":
        # a match's source is before the group or in bytes of the group no run of this pass writes
        owned = np.zeros(HIST + SPAN, dtype=bool)
        for d, _, n in runs:
            owned[HIST + d:HIST + d + n] = True
        for r in runs:
            d, _, n = r
            if not n:
                continue
            choices = [n, n + 1, n + rng.randint(2, 9), d + rng.randint(n, HIST)]
            if d + n <= HIST:
                choices.append(d + n)                           # the source ends exactly at the group's first byte
            for _ in range(64):
                off = rng.choice(choices)
                s = HIST + d - off
                if off >= n and s >= 0 and not owned[s:s + n].any():
                    r[1] = off
                    break
            else:
                r[1] = d + HIST                                 # the history's first byte: always before the group
                if r[1] < n:
                    r[2] = 0
    return {"kind": kind, "runs": runs, "g_align": g_align, "src_align": src_align, "fill": rng.randrange(256)}


def make_cases(seed=7, per=3):
    """per full groups and one sparse group for every kind and pair of alignments."""
    rng = random.Random(seed)
    return [make_case(rng, kind, ga, sa, sparse=(k == per)) for kind in KINDS for ga in range(8) for sa in range(8)
            for k in range(per + 1)]


def total_units(desc, runs):
    """Units of each case's copy as flat_literals / flat_matches count them: 4-byte destination words for literal runs and
    fills, 4-byte pieces of the run for matches.  Above 32 the copy runs two rows per pass (U = 2), else one (U = 1)."""
    out = []
    for d, rr in zip(desc, runs):
        g = int(d[1])
        if d[0] == 2:
            out.append(sum((int(n) + 3) // 4 for _, _, n in rr))
        else:
            out.append(sum(((g + int(p)) % 4 + int(n) + 3) // 4 for p, _, n in rr if n))
    return out


def layout(cases, seed=11):
    """The buffers of a launch: per case a region of HIST history bytes, the group's SPAN bytes and a tail, all random (the
    sentinels); the literal buffer holds each case's literal base at its source alignment."""
    rng = np.random.default_rng(seed)
    region = 64 + HIST + SPAN + 64
    region += -region % 64
    buf = rng.integers(0, 256, size=region * len(cases), dtype=np.uint8)
    lits = rng.integers(0, 256, size=LIT_ROOM * len(cases), dtype=np.uint8)
    desc = np.zeros((len(cases), 4), dtype=np.uint64)
    runs = np.zeros((len(cases), 32, 3), dtype=np.uint32)
    for i, c in enumerate(cases):
        desc[i] = (KINDS.index(c["kind"]), region * i + 64 + HIST + c["g_align"], LIT_ROOM * i + c["src_align"], c["fill"])
        runs[i] = c["runs"]
    return desc, runs, lits, buf


def reference(desc, runs, lits, buf):
    """The expected buffer: each run copied with NumPy slices from the bytes as they were before the launch."""
    out = buf.copy()
    for d, rr in zip(desc, runs):
        kind, g, lbase, fill = (int(x) for x in d)
        for dpos, s, n in (tuple(int(x) for x in r) for r in rr):
            if not n:
                continue
            if kind == 0:
                out[g + dpos:g + dpos + n] = lits[lbase + s:lbase + s + n]
            elif kind == 1:
                out[g + dpos:g + dpos + n] = fill
            else:
                out[g + dpos:g + dpos + n] = buf[g + dpos - s:g + dpos - s + n]
    return out


def serial_model(desc, runs, lits, buf):
    """zstd's sequence execution byte by byte: each run in lane order, every byte read after the bytes before it are written."""
    out = bytearray(buf.tobytes())
    lit = lits.tobytes()
    for d, rr in zip(desc, runs):
        kind, g, lbase, fill = (int(x) for x in d)
        for dpos, s, n in (tuple(int(x) for x in r) for r in rr):
            for k in range(n):
                p = g + dpos + k
                out[p] = lit[lbase + s + k] if kind == 0 else fill if kind == 1 else out[p - s]
    return np.frombuffer(bytes(out), dtype=np.uint8)


# ---------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------
def test_cases_cover_the_plan():
    cases = make_cases()
    lens = {n for c in cases for _, _, n in c["runs"]}
    assert 0 in lens and 127 in lens and len(lens) > 100
    assert {(c["g_align"], c["src_align"]) for c in cases} == {(a, b) for a in range(8) for b in range(8)}
    m = [r for c in cases if c["kind"] == "matches" for r in c["runs"] if r[2]]
    assert any(off == n for _, off, n in m) and any(off == n + 1 for _, off, n in m)
    assert any(off == d + n for d, off, n in m)                  # ends at the group's first byte
    desc, runs, _, _ = layout(cases)
    for d, rr in zip(desc, runs):                                 # neighbouring runs that share a destination word
        g = int(d[1])
        ends = {(g + int(p) + int(n)) // 8 for p, _, n in rr if n}
        starts = {(g + int(p)) // 8 for p, _, n in rr if n}
        if d[0] != 2 and ends & starts:
            break
    else:
        pytest.fail("no case packs two runs into one destination word")
    units = total_units(desc, runs)
    for k in range(len(KINDS)):                                   # both the one-row and the two-row passes of every copy
        u = [x for d, x in zip(desc, units) if d[0] == k]
        assert min(u) <= 32 < max(u), KINDS[k]


def test_reference_agrees_with_a_byte_serial_model():
    desc, runs, lits, buf = layout(make_cases(seed=3, per=1))
    assert np.array_equal(reference(desc, runs, lits, buf), serial_model(desc, runs, lits, buf))


def test_gpu_harness_builds():
    """The harness compiles for sm_100a (without running: that needs a device)."""
    assert build_harness().exec_copy_run


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("seed", [7, 8, 9])
def test_gpu_flat_copies_match_the_serial_copy(seed):
    lib = build_harness()
    desc, runs, lits, buf = layout(make_cases(seed=seed), seed=seed + 100)
    want = reference(desc, runs, lits, buf)
    got = buf.copy()
    e = lib.exec_copy_run(len(desc), desc.ctypes.data, runs.ctypes.data, lits.ctypes.data, lits.size, got.ctypes.data, got.size)
    if e in (35, 100):                                           # cudaErrorInsufficientDriver, cudaErrorNoDevice
        pytest.skip("no CUDA device")
    assert e == 0, f"CUDA error {e}"
    bad = np.nonzero(got != want)[0]
    if bad.size:
        region = buf.size // len(desc)
        i = int(bad[0]) // region
        pytest.fail(f"{bad.size} bytes differ; first at {int(bad[0])}: case {i} kind {KINDS[int(desc[i][0])]} g {int(desc[i][1])} "
                    f"runs {runs[i].tolist()}")
