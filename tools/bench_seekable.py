"""Seekable archives on one GPU: for log text and tick records (--bytes each, 1 GiB by default) in 64 KiB and 1 MiB frames at levels
1 and 3 (with checksums), per shape:
  * compress GB/s of zstdb200_compress_seekable_device (device-resident, CUDA events) and zstdb200_compress_seekable (host to host,
    wall clock);
  * full-range decode GB/s of zstdb200_decompress_seekable_device, next to zstdb200_decompress_batch_device on the same frames at
    the same offsets (the difference is the table's two copies and the check);
  * host-to-host decode of the archive's first --pass-frames frames as ONE item through zstdb200_decompress (one pipeline pass per
    frame) against zstdb200_decompress_seekable of the same archive;
  * median latency of a random 1 MiB range through zstdb200_decompress_seekable_device (wall clock, synchronised).
Rates are content bytes over time; medians of --reps timed repeats after --warmup calls.  The card's name and power limit are read
in the same run.  Prints one JSON line per shape and appends them to --out.

Usage: python tools/bench_seekable.py [--bytes N] [--reps R] [--warmup W] [--out FILE]"""
import argparse
import json
import os
import random
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_dict_compress import card  # noqa: E402


def _events(fn, reps, st):
    """Median ms of fn() between events on st: the device calls enqueue on st, so the events bracket their kernels."""
    import torch
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn()
        b.record(st)
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return statistics.median(out)


def _wall(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(out)


def run_shape(ctx, kind, fs, level, args):
    import torch
    from tools import corpus
    raw = np.ascontiguousarray(corpus.make(kind, args.bytes))
    n = len(raw)
    dev = torch.device("cuda:0")
    t_src = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
    t_src[:n] = torch.from_numpy(raw).to(dev)
    cap = ctx.seekable_bound(n, fs)
    t_arc = torch.zeros(cap + 64, dtype=torch.uint8, device=dev)
    t_size = torch.zeros(1, dtype=torch.int64, device=dev)
    row = {"corpus": kind, "frame": fs, "level": level, "bytes": n}
    st = torch.cuda.Stream(device=dev)
    s = st.cuda_stream

    def dcomp():
        ctx.compress_seekable_device(level, True, fs, t_src.data_ptr(), n, t_arc.data_ptr(), cap, t_size.data_ptr(), stream=s)
    for _ in range(args.warmup):
        dcomp()
    torch.cuda.synchronize()
    ms = _events(dcomp, args.reps, st)
    row["compress_device_gbps"] = round(n / ms / 1e6, 2)
    archive = t_arc[:int(t_size.item())].cpu().numpy().tobytes()
    row["ratio"] = round(n / len(archive), 4)
    host_arc = ctx.compress_seekable(raw, fs, level, True)
    assert host_arc == archive, "host and device archives differ"
    ms = _wall(lambda: ctx.compress_seekable(raw, fs, level, True), args.reps)
    row["compress_host_gbps"] = round(n / ms / 1e6, 2)

    # full-range decode, seekable against the plain batch call on the same frames at the same offsets
    info = ctx.seekable_info(archive)
    nf = info.n_frames
    t_out = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
    t_code = torch.zeros(1, dtype=torch.int32, device=dev)
    alen = len(archive)

    def dseek():
        ctx.decompress_seekable_device(t_out.data_ptr(), 0, n, t_arc.data_ptr(), alen, t_code.data_ptr(), stream=s)
    for _ in range(args.warmup):
        dseek()
    torch.cuda.synchronize()
    assert int(t_code.item()) == 0 and torch.equal(t_out[:n], t_src[:n]), "seekable decode differs"
    ms_seek = _events(dseek, args.reps, st)
    tab = archive[alen - (8 + nf * 12 + 9):]
    ents = np.frombuffer(tab[8:8 + nf * 12], dtype=np.uint32).reshape(nf, 3)
    csz, dsz = ents[:, 0].astype(np.int64), ents[:, 1].astype(np.int64)
    soff = np.concatenate([[0], np.cumsum(csz)[:-1]]).astype(np.int64)
    doff = np.concatenate([[0], np.cumsum(dsz)[:-1]]).astype(np.int64)
    t_soff, t_doff = torch.from_numpy(soff).to(dev), torch.from_numpy(doff).to(dev)
    t_ssz, t_cap = torch.from_numpy(csz.astype(np.int32)).to(dev), torch.from_numpy(dsz.astype(np.int32)).to(dev)
    t_res = torch.zeros(nf, dtype=torch.int32, device=dev)

    def dbatch():
        ctx.decompress_batch_device(t_arc.data_ptr(), t_soff.data_ptr(), t_ssz.data_ptr(), t_out.data_ptr(), t_doff.data_ptr(),
                                    t_cap.data_ptr(), t_res.data_ptr(), nf, stream=s)
    for _ in range(args.warmup):
        dbatch()
    torch.cuda.synchronize()
    assert (t_res.cpu().numpy().view(np.uint32) == dsz).all() and torch.equal(t_out[:n], t_src[:n]), "batch decode differs"
    ms_batch = _events(dbatch, args.reps, st)
    row["decode_seekable_device_gbps"] = round(n / ms_seek / 1e6, 2)
    row["decode_batch_device_gbps"] = round(n / ms_batch / 1e6, 2)

    # the first frames as one item through the existing decoder (a pass per frame) against the seekable call, host to host
    k = min(args.pass_frames, nf)
    part = raw[:min(n, k * fs)]
    small = ctx.compress_seekable(part, fs, level, True)
    out = np.zeros(len(part), dtype=np.uint8)
    res = ctx.decompress_batch([small], [out])
    assert int(res[0]) == len(part) and out.tobytes() == part.tobytes()
    row["one_item_frames"] = k
    row["one_item_decompress_ms"] = round(_wall(lambda: ctx.decompress_batch([small], [out]), args.reps), 3)
    row["one_item_seekable_ms"] = round(_wall(lambda: ctx.decompress_seekable(small, 0, len(part), out=out), args.reps), 3)

    # random 1 MiB ranges, device variant, synchronised
    rng = random.Random(7)
    lat = []
    for i in range(args.ranges + args.warmup):
        a = rng.randrange(n - (1 << 20))
        t0 = time.perf_counter()
        ctx.decompress_seekable_device(t_out.data_ptr(), a, 1 << 20, t_arc.data_ptr(), alen, t_code.data_ptr(), stream=s)
        torch.cuda.synchronize()
        if i >= args.warmup:
            lat.append((time.perf_counter() - t0) * 1e3)
    assert int(t_code.item()) == 0 and torch.equal(t_out[:1 << 20], t_src[a:a + (1 << 20)])
    row["range_1mib_median_ms"] = round(statistics.median(lat), 3)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bytes", type=int, default=1 << 30)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ranges", type=int, default=50)
    ap.add_argument("--pass-frames", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import zstandard_b200 as zb
    info = card()
    ctx = zb.Context(max_batch_bytes=args.bytes)
    lines = []
    for kind in ("log", "tick"):
        for fs in (65536, 1 << 20):
            for level in (1, 3):
                line = json.dumps({**info, **run_shape(ctx, kind, fs, level, args)})
                print(line, flush=True)
                lines.append(line)
    ctx.close()
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
