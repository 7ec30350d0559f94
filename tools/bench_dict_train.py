"""Dictionary training on the GPU against single-threaded ZDICT_trainFromBuffer: one JSON line per sample-set size.

4 KiB log messages (tools/corpus.py), 32 KiB capacity, default parameters (k searched as ZDICT_trainFromBuffer does).  Reports
the wall time of the synchronous zstdb200_train_dictionary call after one warm-up call, ZDICT's time on this host, the k each
chose, and the compressed size of 1024 held-out messages with each dictionary (libzstd level 3; this library at levels 1-3)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return name, power
    except Exception:
        return "unknown", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes-mib", default="32,256")
    ap.add_argument("--capacity", type=int, default=32768)
    a = ap.parse_args()
    import numpy as np
    import zstandard_b200 as zb
    from tools import corpus, zstd_ref
    name, power = gpu_info()
    ctx = zb.Context(max_batch_bytes=64 << 20)
    for mib in [int(x) for x in a.sizes_mib.split(",")]:
        total = mib << 20
        text = corpus.log(total + (4 << 20)).tobytes()
        samples = [text[i:i + 4096] for i in range(0, total, 4096)]
        held = [text[total + 4096 * i:total + 4096 * (i + 1)] for i in range(1024)]
        ctx.train_dictionary(samples, a.capacity)                            # warm-up
        t0 = time.perf_counter(); ours = ctx.train_dictionary(samples, a.capacity); t_gpu = time.perf_counter() - t0
        k_gpu = ctx.last_train_params.k
        t0 = time.perf_counter(); theirs = zstd_ref.train_dict(samples, a.capacity); t_cpu = time.perf_counter() - t0
        raw = sum(len(m) for m in held)

        def ours_size(d, lv):
            ctx.load_dictionary(d)
            dsts = [np.zeros(zb.ZStdCompress.CompressBound(4096), dtype=np.uint8) for _ in held]
            res = ctx.compress_batch_using_dict(held, dsts, level=lv, checksum=False)
            ctx.load_dictionary(None)
            return int(sum(int(r) for r in res))
        row = {"samples_mib": mib, "capacity": a.capacity, "gpu_train_s": round(t_gpu, 4), "zdict_train_s": round(t_cpu, 4),
               "k_gpu": k_gpu, "dict_bytes_gpu": len(ours), "dict_bytes_zdict": len(theirs)}
        for tag, d in (("gpu", ours), ("zdict", theirs)):
            row[f"ratio_libzstd3_{tag}"] = round(raw / sum(len(zstd_ref.compress_with_dict(m, d, 3, False)) for m in held), 4)
            for lv in (1, 2, 3):
                row[f"ratio_ours{lv}_{tag}"] = round(raw / ours_size(d, lv), 4)
        row.update({"gpu": name, "power_limit": power})
        print(json.dumps(row), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
