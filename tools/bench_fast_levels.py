"""Negative compression levels on one GPU: zstdb200_compress_batch_device at levels 1, -1, -2, -3, -5 and -7 on log text and tick
records in 4 KiB and 128 KiB chunks, plus level 1 and -1 with a 32 KiB ZDICT dictionary on 4 KiB log messages.  Device-resident
input and output, no checksum.  Per shape the levels are alternated: each of --reps rounds times --steps calls of every level
with CUDA events (after --warmup calls each), and the median round is reported.  A separate zstdb200_compress_batch_device_timed
call gives the per-kernel times.  Also recorded: the compression ratio, libzstd 1.5.5's ratio at the same level, libzstd's
all-core CPU throughput (zstd_ref.compress_chunks, wall clock), and the card's name and power limit read in the same run.
Prints one JSON line per shape (and appends them to --out).

Usage: python tools/bench_fast_levels.py [--bytes N] [--steps K] [--warmup W] [--reps R] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_dict_compress import card  # noqa: E402

LEVELS = (1, -1, -2, -3, -5, -7)
DICT_LEVELS = (1, -1)


def run_shape(ctx, kind, chunk, nbytes, levels, args, dictionary=None):
    import torch
    import zstandard_b200 as zb
    from tools import corpus, zstd_ref
    raw = corpus.make(kind, nbytes)
    n = len(raw) // chunk
    total = n * chunk
    raw = np.ascontiguousarray(raw[:total])
    ctx.load_dictionary(dictionary)
    bound = (zb.ZStdCompress.CompressBound(chunk) + 15) // 16 * 16
    dev = torch.device("cuda:0")
    t_src = torch.zeros(total + 64, dtype=torch.uint8, device=dev)
    t_src[:total] = torch.from_numpy(raw).to(dev)
    t_dst = torch.zeros(n * bound, dtype=torch.uint8, device=dev)
    t_soff = torch.arange(n, dtype=torch.int64, device=dev) * chunk
    t_doff = torch.arange(n, dtype=torch.int64, device=dev) * bound
    t_ssz = torch.full((n,), chunk, dtype=torch.int32, device=dev)
    t_cap = torch.full((n,), bound, dtype=torch.int32, device=dev)
    t_res = torch.zeros(n, dtype=torch.int32, device=dev)
    st = torch.cuda.Stream(device=dev)
    dargs = (t_src.data_ptr(), t_soff.data_ptr(), t_ssz.data_ptr(), t_dst.data_ptr(), t_doff.data_ptr(), t_cap.data_ptr(), t_res.data_ptr(), n)
    fn = ctx.compress_batch_device_using_dict if dictionary else ctx.compress_batch_device

    def check():
        res = t_res.cpu().numpy().view(np.uint32)
        assert (res < 0xFFFFFF88).all(), "compress failed"
        out = t_dst.cpu().numpy()
        for k in range(0, n, max(1, n // 64)):
            f = out[k * bound:k * bound + int(res[k])].tobytes()
            want = raw[k * chunk:(k + 1) * chunk].tobytes()
            got = zstd_ref.decompress_with_dict(f, chunk, dictionary) if dictionary else zstd_ref.decompress(f, chunk)
            assert got == want, "frame does not round-trip"
        return int(res.astype(np.int64).sum())

    rows = {lv: {} for lv in levels}
    for lv in levels:
        for _ in range(args.warmup):
            fn(lv, False, *dargs, stream=st.cuda_stream)
        torch.cuda.synchronize()
        rows[lv]["ratio"] = round(total / check(), 4)
        if not dictionary:                                   # the timed entry point never uses the dictionary
            ms = ctx.compress_batch_device_timed(lv, False, *dargs, stream=st.cuda_stream)
            rows[lv]["kernel_ms"] = {k: round(v, 3) for k, v in ms.items()}
    times = {lv: [] for lv in levels}
    for _ in range(args.reps):                               # levels alternated round by round
        for lv in levels:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(st):
                ev0.record(st)
                for _ in range(args.steps):
                    fn(lv, False, *dargs, stream=st.cuda_stream)
                ev1.record(st)
            torch.cuda.synchronize()
            times[lv].append(ev0.elapsed_time(ev1) / args.steps)
    threads = max(1, os.cpu_count() or 1)
    for lv in levels:
        ms = statistics.median(times[lv])
        rows[lv]["gbps"] = round(total / ms / 1e6, 2)
        rows[lv]["ms"] = round(ms, 3)
        rows[lv]["ms_rounds"] = [round(t, 3) for t in times[lv]]
        t0 = time.perf_counter()
        _, off = zstd_ref.compress_chunks(raw, chunk, level=lv, checksum=False, threads=threads, dictionary=dictionary)
        cpu_s = time.perf_counter() - t0
        rows[lv]["libzstd_ratio"] = round(total / int(off[-1]), 4)
        rows[lv]["libzstd_cpu_gbps"] = round(total / cpu_s / 1e9, 3)
    ctx.load_dictionary(None)
    return {"corpus": kind, "chunk": chunk, "bytes": total, "dictionary_bytes": len(dictionary) if dictionary else 0,
            "libzstd_threads": threads, "levels": {str(lv): rows[lv] for lv in levels}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bytes", type=int, default=256 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import zstandard_b200 as zb
    from tools import corpus, zstd_ref
    info = card()
    what = ("zstdb200_compress_batch_device(_using_dict), device-resident, no checksum; median of %d alternated rounds of %d calls "
            "after %d warm-ups" % (args.reps, args.steps, args.warmup))
    ctx = zb.Context(max_batch_bytes=args.bytes + (16 << 20))
    head = corpus.make("log", 16 << 20).tobytes()
    dictionary = zstd_ref.train_dict([head[i:i + 4096] for i in range(0, len(head), 4096)][:4096], 32768)
    shapes = [("log", 4096, LEVELS, None), ("log", 131072, LEVELS, None), ("tick", 4096, LEVELS, None),
              ("tick", 131072, LEVELS, None), ("log", 4096, DICT_LEVELS, dictionary)]
    lines = []
    for kind, chunk, levels, d in shapes:
        r = {"what": what, **info, **run_shape(ctx, kind, chunk, args.bytes, levels, args, d)}
        line = json.dumps(r)
        print(line, flush=True)
        lines.append(line)
    ctx.close()
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
