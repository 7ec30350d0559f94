"""Dictionary compression on one GPU: zstdb200_compress_batch_device_using_dict against zstdb200_compress_batch_device on the
same data, the dictionary-decode shape of tools/sweep_configs.sh (4 KiB log messages, a 32 KiB dictionary trained by ZDICT on
the head of the corpus).  Device-resident input and output, CUDA events around `--steps` calls after `--warmup` calls, the two
paths alternated level by level.  Prints one JSON line (and appends it to --out): GB/s of uncompressed input per level with
and without the dictionary, the compression ratios, libzstd 1.5.5's ratios with the same dictionary and level, and the card's
name and power limit read in the same run.

Usage: python tools/bench_dict_compress.py [--bytes N] [--steps K] [--warmup W] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"] = float(q[0]); info["sm_max_mhz"] = float(q[1])
    except Exception as e:                                   # reported, not guessed
        info["power_limit_w"] = None; info["power_limit_error"] = str(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bytes", type=int, default=256 << 20)
    ap.add_argument("--chunk", type=int, default=4096)
    ap.add_argument("--dict-bytes", type=int, default=32768)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import zstandard_b200 as zb
    from tools import corpus, zstd_ref
    raw = corpus.make("log", args.bytes)
    total, chunk = len(raw), args.chunk
    n = total // chunk
    total = n * chunk
    head = raw[:min(total, 16 << 20)].tobytes()
    dictionary = zstd_ref.train_dict([head[i:i + chunk] for i in range(0, len(head), chunk)][:4096], args.dict_bytes)
    ctx = zb.Context(max_batch_bytes=total + (16 << 20))
    ctx.load_dictionary(dictionary)
    bound = (zb.ZStdCompress.CompressBound(chunk) + 15) // 16 * 16
    dev = torch.device("cuda:0")
    t_src = torch.zeros(total + 64, dtype=torch.uint8, device=dev)
    t_src[:total] = torch.from_numpy(np.ascontiguousarray(raw[:total])).to(dev)
    t_dst = torch.zeros(n * bound, dtype=torch.uint8, device=dev)
    t_soff = torch.arange(n, dtype=torch.int64, device=dev) * chunk
    t_doff = torch.arange(n, dtype=torch.int64, device=dev) * bound
    t_ssz = torch.full((n,), chunk, dtype=torch.int32, device=dev)
    t_cap = torch.full((n,), bound, dtype=torch.int32, device=dev)
    t_res = torch.zeros(n, dtype=torch.int32, device=dev)
    st = torch.cuda.Stream(device=dev)
    dargs = (t_src.data_ptr(), t_soff.data_ptr(), t_ssz.data_ptr(), t_dst.data_ptr(), t_doff.data_ptr(), t_cap.data_ptr(), t_res.data_ptr(), n)

    def call(level, use_dict):
        fn = ctx.compress_batch_device_using_dict if use_dict else ctx.compress_batch_device
        fn(level, True, *dargs, stream=st.cuda_stream)

    def check(level, use_dict):
        res = t_res.cpu().numpy().view(np.uint32)
        assert (res < 0xFFFFFF88).all(), "compress failed"
        out = t_dst.cpu().numpy()
        for k in range(0, n, max(1, n // 64)):
            f = out[k * bound:k * bound + int(res[k])].tobytes()
            want = raw[k * chunk:(k + 1) * chunk].tobytes()
            got = zstd_ref.decompress_with_dict(f, chunk, dictionary) if use_dict else zstd_ref.decompress(f, chunk)
            assert got == want, "frame does not round-trip"
        return int(res.astype(np.int64).sum())

    result = {"what": "zstdb200_compress_batch_device(_using_dict), %d x %d B log messages, %d-byte trained dictionary, checksum on, "
                      "device-resident, CUDA events over %d calls after %d warm-ups" % (n, chunk, len(dictionary), args.steps, args.warmup),
              "bytes": total, **card(), "levels": {}}
    for level in (1, 2, 3):
        row = {}
        for use_dict in (False, True):                     # both paths on the same data, one after the other per level
            for _ in range(max(3, args.warmup)):
                call(level, use_dict)
            torch.cuda.synchronize()
            size = check(level, use_dict)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(st):
                ev0.record(st)
                for _ in range(args.steps):
                    call(level, use_dict)
                ev1.record(st)
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / args.steps
            key = "dict" if use_dict else "plain"
            row[key + "_gbps"] = round(total / ms / 1e6, 2)
            row[key + "_ms"] = round(ms, 3)
            row[key + "_ratio"] = round(total / size, 4)
        _, off = zstd_ref.compress_chunks(raw[:total], chunk, level=level, checksum=True, threads=max(1, os.cpu_count() or 1), dictionary=dictionary)
        row["libzstd_dict_ratio"] = round(total / int(off[-1]), 4)
        _, off = zstd_ref.compress_chunks(raw[:total], chunk, level=level, checksum=True, threads=max(1, os.cpu_count() or 1))
        row["libzstd_plain_ratio"] = round(total / int(off[-1]), 4)
        row["dict_speed_vs_plain"] = round(row["dict_gbps"] / row["plain_gbps"], 3)
        result["levels"][str(level)] = row
    ctx.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
