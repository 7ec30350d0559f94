#!/usr/bin/env python3
"""bench.py — headline benchmark of libzstdb200 (BASELINE.json: GB/s uncompressed, 64 KiB frames).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload decode64k|compress128k]
                    [--corpus log|tick|random|mixed] [--chunk BYTES] [--level 1..3] [--bytes N] [--dictionary BYTES]
                    [--no-extras] [--no-cpu-baseline] [--dump-outputs DIR]

One process per GPU (under torchrun for N > 1: RANK/LOCAL_RANK/WORLD_SIZE from the env).  Frames are independent,
so ranks shard the work with no data-path collective ("scaling": "weak": every rank processes --bytes of its own
synthetic data); torch.distributed is used only for the barrier and the max-over-ranks time.

A step = one pass of the hot path over one batch:
  decode64k    (default, BASELINE.json configs[1]) decodes --bytes (1 GiB) of libzstd level-3 compressed log text held
               as 64 KiB frames with XXH64 checksums
  compress128k (configs[2]) compresses --bytes of log text in 128 KiB chunks at --level with XXH64 checksums
Reported:
  value         device-resident pipeline: inputs and outputs already in HBM, CUDA events on the launching stream
  e2e           the same work through the host-buffer C-ABI call (pinned host memory -> H2D -> kernels -> D2H)
  roofline      algorithmic bytes (bytes in + bytes out of the codec) / duration of the dominant kernel; `traffic` = that
                kernel's DRAM bytes per launch from the committed ncu capture of this command (profiles/traffic.json)
The default line (decode64k, log text, no --chunk) also carries
  compress        BASELINE.json configs[2]: levels 1-3 on the same corpus in 128 KiB chunks — value, e2e, our / libzstd ratio,
                  per-kernel ms, roofline fractions (the reference has no compressor: the ratio band is unpinned by it)
  e2e_pageable    the same C-ABI call on pageable caller memory (what a managed byte[] is): one array pair / one array per frame
  single_call_us  median latency of zstdb200_decompress on one 64 KiB frame
  multi_block     (N = 1) tick records as 256 KiB / 1 MiB frames (2 / 8 blocks each, configs[4]'s large end): value, e2e, per-kernel ms
  e2e_single_ctx  (N > 1, under torchrun) rank 0 alone driving ONE context over all N devices on N x the workload
The other BASELINE.json configs are the same two workloads with other shapes: --corpus mixed (configs[3]), --corpus tick
--chunk 4096..1048576 (configs[4]); profiles/ holds the lines measured for them.
  cpu_baseline  decode: the oracle (C++ port of the reference decoder; the C# reference cannot run in this image), with
                libzstd 1.5.5's own decoder beside it as `cpu_baseline_libzstd`; compress: libzstd 1.5.5 (the reference
                has no compressor) — all host cores in every case
`--impl reference` times that CPU baseline alone, rank 0 only, as the reference arm.

--dump-outputs DIR writes what the device-resident arm returned to its caller in the last timed step (rank 0), so that two
builds can be compared output for output on identical inputs (the corpus and libzstd's frames are deterministic):
  result.npy     float64, the result code of every item (bytes written, or the error code)
  dst.npy        float32, one row of dst_stride bytes per sampled item: its destination bytes, zero past its result
  dst_items.npy  float64, the sampled items: np.random.default_rng(0).permutation(n)[:k] sorted, k = as many rows as fit
                 in 32 MiB
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: no __pycache__ next to the imported modules

CHUNK = {"decode64k": 65536, "compress128k": 131072}
METRIC = {"decode64k": "decompress_GBps_uncompressed", "compress128k": "compress_GBps_uncompressed"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="decode64k", choices=list(CHUNK))
    ap.add_argument("--bytes", type=int, default=1 << 30, help="uncompressed bytes per GPU per step")
    ap.add_argument("--corpus", default="log", choices=["log", "tick", "random", "mixed"])
    ap.add_argument("--level", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=0, help="frame / chunk size in bytes (default: the workload's 64 KiB / 128 KiB)")
    ap.add_argument("--dictionary", type=int, default=0, help="decode only: frames compressed with a dictionary of this many bytes trained "
                    "(ZDICT) on the head of the corpus, decoded through zstdb200_load_dictionary (SURVEY 8f-3)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the compress block, the pageable / single-call / single-context measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as .npy files to DIR (see the docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    return args


def recorded_traffic(workload_key, kernel):
    """DRAM bytes per launch of `kernel` from the ncu --set full capture of this bench command (profiles/traffic.json,
    written by tools/ncu_traffic.py from the committed capture); None when no capture exists for this workload."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    rec = json.load(open(p)).get(workload_key, {}).get(kernel)
    return int(rec["dram_bytes"]) if rec else None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (B200_PROFILING.md clocks line, via NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------------
# workload: host-side description of one step.  `src` is the codec's input, `dst` its output.
# ----------------------------------------------------------------------------------------------------------
def prepare(args, rank, workload=None, level=None, raw=None):
    from tools import corpus, zstd_ref
    import zstandard_b200 as zb
    workload = workload or args.workload
    level = level or args.level
    chunk = (args.chunk if workload == args.workload else 0) or CHUNK[workload]
    if raw is None:
        raw = corpus.make(args.corpus, args.bytes, shard=rank)
    total = len(raw)
    n = (total + chunk - 1) // chunk
    raw_off = np.arange(n + 1, dtype=np.uint64) * chunk
    raw_off[-1] = total
    w = {"raw": raw, "chunk": chunk, "n": n, "total": total, "kind": workload, "level": level, "dictionary": None}
    if args.dictionary and workload == "decode64k":
        head = raw[:min(total, 16 << 20)].tobytes()
        w["dictionary"] = zstd_ref.train_dict([head[i:i + chunk] for i in range(0, len(head), chunk)][:4096], args.dictionary)
        plain, poff = zstd_ref.compress_chunks(raw, chunk, level=level, checksum=True, threads=max(1, os.cpu_count() or 1))
        w["plain_compressed_bytes"] = int(poff[-1])
    blob, off = zstd_ref.compress_chunks(raw, chunk, level=level, checksum=True, threads=max(1, os.cpu_count() or 1), dictionary=w["dictionary"])
    w["ref_compressed_bytes"] = int(off[-1])
    if workload == "decode64k":
        w.update(src=blob, src_off=off, dst_cap=np.diff(raw_off).astype(np.uint32), dst_stride=chunk)
    else:
        bound = (zb.ZStdCompress.CompressBound(chunk) + 15) // 16 * 16
        w.update(src=raw, src_off=raw_off, dst_cap=np.full(n, bound, dtype=np.uint32), dst_stride=bound)
    return w


def workload_config(args, w):
    if w["kind"] == "decode64k":
        what = (f"decode{w['chunk'] // 1024}k: batched decompression of {w['total']} B/GPU of libzstd-1.5.5 level-{w['level']} {args.corpus} text held as "
                f"{w['chunk'] // 1024} KiB independent frames with XXH64 checksums")
    else:
        what = (f"compress{w['chunk'] // 1024}k: batched level-{w['level']} compression of {w['total']} B/GPU of {args.corpus} text in "
                f"{w['chunk'] // 1024} KiB chunks, one frame each, with XXH64 checksums")
    extra = {}
    if w.get("dictionary"):
        what += f", compressed with a {len(w['dictionary'])}-byte trained dictionary (ZSTD_decompress_usingDict path)"
        extra = {"dictionary_bytes": len(w["dictionary"]), "libzstd_ratio_without_dictionary": round(w["total"] / w["plain_compressed_bytes"], 4)}
    return {**extra, "workload": what, "frames_per_gpu": w["n"], "libzstd_compressed_bytes_per_gpu": w["ref_compressed_bytes"],
            "libzstd_ratio": round(w["total"] / w["ref_compressed_bytes"], 4),
            "l2": "inputs+outputs per step exceed the 126 MB L2 (no flush needed)", "sharding": "by frame, no collective"}


class CpuBaseline:
    """All-core CPU arm: oracle batch decode (decode64k) or libzstd compress (compress128k)."""

    def __init__(self, args, w):
        self.w, self.args = w, args
        self.cores = os.cpu_count() or 1
        if w["kind"] == "decode64k":
            from tests import helpers
            self.lib = helpers.Oracle().lib
            n, total = w["n"], w["total"]
            self.out = np.zeros(total, dtype=np.uint8)
            off = w["src_off"]
            bs, bd = w["src"].ctypes.data, self.out.ctypes.data
            self.sp = (ctypes.c_void_p * n)(*[bs + int(off[i]) for i in range(n)])
            self.dp = (ctypes.c_void_p * n)(*[bd + i * w["chunk"] for i in range(n)])
            self.ss = np.diff(off).astype(np.uint32)
            self.dc = w["dst_cap"].copy()
            self.res = np.zeros(n, dtype=np.uint32)
            self.lib.oracle_decompress_batch.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_uint64, ctypes.c_int]
            self.lib.oracle_decompress_batch.restype = None
            self.kind, self.what = "port", "oracle = C++ restatement of the reference C# decoder, static frame partition over all cores"
            # second CPU baseline (SURVEY.md §8d ii): libzstd 1.5.5 ZSTD_decompress on all cores (tools/zstd_mt.c)
            self.zmt = None
            zp = os.path.join(ROOT, "tools", "_build", "libzstdmt.so")
            if os.path.exists(zp):
                self.zmt = ctypes.CDLL(zp)
                self.zmt.zmt_decompress.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64,
                                                    ctypes.c_uint64, ctypes.c_int]
        else:
            self.kind, self.what = "port", ("libzstd 1.5.5 ZSTD_compress2 (the reference ships no compressor; libzstd is the stand-in "
                                             "comparator), one context per core")

    def run(self):
        """-> (seconds, uncompressed bytes processed)"""
        w = self.w
        t = time.perf_counter()
        if w["kind"] == "decode64k":
            self.lib.oracle_decompress_batch(self.sp, self.ss.ctypes.data, self.dp, self.dc.ctypes.data, self.res.ctypes.data, w["n"], self.cores)
            dt = time.perf_counter() - t
            assert (self.res == self.dc).all(), "oracle failed to decode the workload"
        else:
            from tools import zstd_ref
            zstd_ref.compress_chunks(w["raw"], w["chunk"], level=w["level"], checksum=True, threads=self.cores)
            dt = time.perf_counter() - t
        return dt, w["total"]


def libzstd_decode_baseline(cb):
    """-> {"value": GB/s, ...} of libzstd's own decoder on all cores over the same frames, or None."""
    if getattr(cb, "zmt", None) is None:
        return None
    w = cb.w
    off = np.ascontiguousarray(w["src_off"], dtype=np.uint64)
    call = lambda: cb.zmt.zmt_decompress(w["src"].ctypes.data, off.ctypes.data, w["n"], cb.out.ctypes.data, w["chunk"], w["total"], cb.cores)
    if call() != 0:
        return None
    tt, runs = 0.0, 0
    while tt < 1.5 and runs < 20:
        t = time.perf_counter()
        call()
        tt += time.perf_counter() - t
        runs += 1
    return {"value": round(w["total"] * runs / tt / 1e9, 3), "unit": "GB/s", "cores": cb.cores, "kind": "libzstd 1.5.5 ZSTD_decompress",
            "sample": f"{runs} pass(es) over the full step"}


def run_reference(args, rank):
    if rank != 0:
        return
    w = prepare(args, 0)
    cb = CpuBaseline(args, w)
    for _ in range(args.warmup):
        cb.run()
    t = 0.0
    for _ in range(args.steps):
        dt, nbytes = cb.run()
        t += dt
    gbs = nbytes * args.steps / t / 1e9
    line = {"impl": "reference", "metric": METRIC[args.workload], "value": round(gbs, 3), "unit": "GB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * t / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(args, w),
            "cpu_baseline": {"value": round(gbs, 3), "unit": "GB/s", "cores": cb.cores, "kind": cb.kind,
                             "sample": f"full step ({w['n']} frames, {nbytes} B) x {args.steps} steps; {cb.what}"},
            "e2e": {"value": round(gbs, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


class Gpu:
    """One rank's device, context and (optional) process group."""

    def __init__(self, args):
        import torch
        import zstandard_b200 as zb
        self.torch, self.zb = torch, zb
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.lib = zb.load_library()
        self.ctx = zb.Context(devices=[self.local], max_batch_bytes=max(args.bytes, 1 << 20))

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def barrier(self):
        if self.dist:
            self.dist.barrier()


DUMP_ROW_BYTES = 32 << 20      # float32 rows of dst.npy; result.npy and dst_items.npy come on top (64 MB in all at most)


def dump_outputs(out_dir, w, t_dst, t_res):
    """--dump-outputs: result codes of every item and the destination bytes of a seeded sample of items (docstring)."""
    import torch
    n, stride = w["n"], w["dst_stride"]
    res = t_res.cpu().numpy().view(np.uint32)
    k = max(1, min(n, DUMP_ROW_BYTES // (4 * stride)))
    items = np.sort(np.random.default_rng(0).permutation(n)[:k])
    rows = t_dst[:n * stride].view(n, stride)[torch.from_numpy(items).to(t_dst.device)].cpu().numpy()
    written = np.where(res[items] <= stride, res[items], 0)          # an error code writes nothing
    rows[np.arange(stride)[None, :] >= written[:, None].astype(np.int64)] = 0
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "result.npy"), res.astype(np.float64))
    np.save(os.path.join(out_dir, "dst.npy"), rows.astype(np.float32))
    np.save(os.path.join(out_dir, "dst_items.npy"), items.astype(np.float64))


def measure(g, args, w, steps, warmup, sampler=None, extras=False, dump=None):
    """One workload on this rank's GPU: device-resident pipeline (CUDA events, max over ranks), per-kernel times, and the
    host-buffer C-ABI call from pinned memory.  extras: also pageable caller memory and the single-item call (decode).
    dump: a directory for the outputs of the last timed step (dump_outputs)."""
    torch, ctx, lib, dev = g.torch, g.ctx, g.lib, g.dev
    n, total, decode, level = w["n"], w["total"], w["kind"] == "decode64k", w["level"]
    src_bytes = int(w["src_off"][-1])
    dst_span = n * w["dst_stride"]
    # ---------------- device-resident arm ----------------
    t_src = torch.empty(src_bytes + 64, dtype=torch.uint8, device=dev)
    t_src[:src_bytes] = torch.from_numpy(w["src"]).to(dev)
    t_dst = torch.zeros(dst_span + 64, dtype=torch.uint8, device=dev)
    soff = w["src_off"][:-1].astype(np.int64)
    ssz = np.diff(w["src_off"]).astype(np.int32)
    doff = np.arange(n, dtype=np.int64) * w["dst_stride"]
    dcap = w["dst_cap"].view(np.int32)
    t_soff, t_ssz = torch.from_numpy(soff).to(dev), torch.from_numpy(ssz).to(dev)
    t_doff, t_dcap = torch.from_numpy(doff).to(dev), torch.from_numpy(dcap.copy()).to(dev)
    t_res = torch.zeros(n, dtype=torch.int32, device=dev)
    # a non-default stream: handle 0 would mean "the context's own stream" to the C ABI
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    dargs = (t_src.data_ptr(), t_soff.data_ptr(), t_ssz.data_ptr(), t_dst.data_ptr(), t_doff.data_ptr(), t_dcap.data_ptr(),
             t_res.data_ptr(), n)

    def step_device():
        if decode:
            ctx.decompress_batch_device(*dargs, stream=stream)
        else:
            ctx.compress_batch_device(level, True, *dargs, stream=stream)

    def verify(res_u32, out_bytes):
        """what is being timed must be right: decode -> the corpus; compress -> frames an independent decoder accepts"""
        if decode:
            assert (res_u32 == w["dst_cap"]).all(), "decode failed on the bench workload"
            assert (out_bytes[:total] == w["raw"]).all(), "decoded bytes differ from the corpus"
            return None
        from tools import zstd_ref
        assert (res_u32 < 0xFFFFFF88).all(), "compress failed on the bench workload"
        stride = w["dst_stride"]
        for k in range(0, n, max(1, n // 64)):
            f = out_bytes[k * stride:k * stride + int(res_u32[k])].tobytes()
            lo = k * w["chunk"]
            assert zstd_ref.decompress(f, int(ssz[k])) == w["raw"][lo:lo + int(ssz[k])].tobytes(), "frame does not round-trip"
        return int(res_u32.astype(np.int64).sum())

    for _ in range(max(3, warmup)):
        step_device()
    torch.cuda.synchronize()
    our_compressed = verify(t_res.cpu().numpy().view(np.uint32), t_dst.cpu().numpy())

    if sampler:
        sampler.start()
    l0 = ctx.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g.barrier()
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        step_device()
    ev1.record()
    torch.cuda.synchronize()
    g.barrier()
    ms = g.max_over_ranks(ev0.elapsed_time(ev1))
    launches = ctx.kernel_launches - l0
    if dump:
        dump_outputs(dump, w, t_dst, t_res)

    # per-kernel device times (CUDA events between the kernels, separate synchronised runs)
    kms = {}
    reps = max(3, steps)
    for _ in range(reps):
        per = ctx.decompress_batch_device_timed(*dargs, stream=stream) if decode else ctx.compress_batch_device_timed(level, True, *dargs, stream=stream)
        for k, v in per.items():
            kms[k] = kms.get(k, 0.0) + v / reps
    del t_src, t_dst

    # ---------------- end-to-end arm: host buffers through the C ABI ----------------
    u32p = ctypes.POINTER(ctypes.c_uint32)
    ss_u, dc_u, res_u = ssz.view(np.uint32).copy(), w["dst_cap"].copy(), np.zeros(n, dtype=np.uint32)

    def host_call(sp, dp, cnt=n):
        if decode:
            rc = lib.zstdb200_decompress_batch(ctx.handle, sp, ss_u.ctypes.data_as(u32p), dp, dc_u.ctypes.data_as(u32p),
                                               res_u.ctypes.data_as(u32p), cnt)
        else:
            rc = lib.zstdb200_compress_batch(ctx.handle, level, 1, sp, ss_u.ctypes.data_as(u32p), dp, dc_u.ctypes.data_as(u32p),
                                             res_u.ctypes.data_as(u32p), cnt)
        assert rc == 0, ctx.last_error()

    def timed_host(sp, dp, dst_view, k_steps):
        for _ in range(max(1, min(warmup, 2))):
            host_call(sp, dp)
        verify(res_u, dst_view)
        g.barrier()
        t0 = time.perf_counter()
        for _ in range(k_steps):
            host_call(sp, dp)
        return g.max_over_ranks(time.perf_counter() - t0)

    h_src = lib.zstdb200_host_alloc(src_bytes + 64)
    h_dst = lib.zstdb200_host_alloc(dst_span + 64)
    ctypes.memmove(h_src, w["src"].ctypes.data, src_bytes)
    sp = (ctypes.c_void_p * n)(*[h_src + int(w["src_off"][i]) for i in range(n)])
    dp = (ctypes.c_void_p * n)(*[h_dst + i * w["dst_stride"] for i in range(n)])
    got = np.ctypeslib.as_array(ctypes.cast(h_dst, ctypes.POINTER(ctypes.c_uint8)), shape=(dst_span,))
    e2e_s = timed_host(sp, dp, got, steps)
    lib.zstdb200_host_free(h_src)
    lib.zstdb200_host_free(h_dst)

    out = {"ms": ms, "steps": steps, "launches": int(launches), "kernel_ms": kms, "our_compressed": our_compressed, "e2e_s": e2e_s,
           "src_bytes": src_bytes, "n": n, "total": total}
    if extras and decode:
        # the memory a managed caller really has: pageable (a `fixed` byte[] is pinned for the GC, not for CUDA,
        # ZStdDecompress.cs:2182-2186) — one contiguous array pair, and one separate array per frame
        p_dst = np.zeros(dst_span + 64, dtype=np.uint8)
        sp2 = (ctypes.c_void_p * n)(*[w["src"].ctypes.data + int(w["src_off"][i]) for i in range(n)])
        dp2 = (ctypes.c_void_p * n)(*[p_dst.ctypes.data + i * w["dst_stride"] for i in range(n)])
        k_steps = max(1, min(steps, 3))
        out["e2e_pageable_s"] = timed_host(sp2, dp2, p_dst, k_steps) / k_steps
        srcs = [w["src"][int(w["src_off"][i]):int(w["src_off"][i + 1])].copy() for i in range(n)]
        dsts = [np.zeros(int(w["dst_cap"][i]), dtype=np.uint8) for i in range(n)]
        sp3 = (ctypes.c_void_p * n)(*[a.ctypes.data for a in srcs])
        dp3 = (ctypes.c_void_p * n)(*[a.ctypes.data for a in dsts])
        host_call(sp3, dp3)
        assert all((dsts[i] == w["raw"][i * w["chunk"]:i * w["chunk"] + len(dsts[i])]).all() for i in range(0, n, max(1, n // 64)))
        t0 = time.perf_counter()
        for _ in range(k_steps):
            host_call(sp3, dp3)
        out["e2e_scattered_s"] = g.max_over_ranks(time.perf_counter() - t0) / k_steps
        # one frame per call: ZStdDecompress.Decompress(byte[], uint, byte[], uint) as the shim issues it
        lib.zstdb200_decompress.restype = ctypes.c_uint32
        lib.zstdb200_decompress.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_uint32]
        one = []
        for k in range(24):
            i = (k * 37) % n
            t0 = time.perf_counter()
            r = lib.zstdb200_decompress(ctx.handle, dsts[i].ctypes.data, len(dsts[i]), srcs[i].ctypes.data, len(srcs[i]))
            one.append(time.perf_counter() - t0)
            assert r == len(dsts[i])
        out["single_call_us"] = float(np.median(one[4:]) * 1e6)
    return out


def single_context_all_devices(g, args, w, steps):
    """Rank 0 drives ONE context over all N devices of the box (the library's own sharding: sub-batches dealt to one
    host thread per device, api.cu run_host_batch) on N x the per-GPU workload; verified against the corpus."""
    zb, lib = g.zb, g.lib
    N, n, total = g.world, w["n"], w["total"]
    src_bytes, stride = int(w["src_off"][-1]), w["dst_stride"]
    ctx = zb.Context(devices=list(range(N)), max_batch_bytes=max(total, 1 << 20))
    try:
        span_s = (src_bytes + 63) // 64 * 64
        h_src = lib.zstdb200_host_alloc(N * span_s + 64)
        h_dst = lib.zstdb200_host_alloc(N * n * stride + 64)
        for k in range(N):
            ctypes.memmove(h_src + k * span_s, w["src"].ctypes.data, src_bytes)
        sp = (ctypes.c_void_p * (N * n))(*[h_src + k * span_s + int(w["src_off"][i]) for k in range(N) for i in range(n)])
        dp = (ctypes.c_void_p * (N * n))(*[h_dst + (k * n + i) * stride for k in range(N) for i in range(n)])
        ss = np.tile(np.diff(w["src_off"]).astype(np.uint32), N)
        dc = np.tile(w["dst_cap"], N)
        res = np.zeros(N * n, dtype=np.uint32)
        u32p = ctypes.POINTER(ctypes.c_uint32)
        call = lambda: lib.zstdb200_decompress_batch(ctx.handle, sp, ss.ctypes.data_as(u32p), dp, dc.ctypes.data_as(u32p), res.ctypes.data_as(u32p), N * n)
        assert call() == 0, ctx.last_error()
        assert (res == dc).all()
        got = np.ctypeslib.as_array(ctypes.cast(h_dst, ctypes.POINTER(ctypes.c_uint8)), shape=(N * n * stride,))
        for k in range(N):
            assert (got[k * n * stride:k * n * stride + total] == w["raw"]).all(), "single-context decode differs from the corpus"
        t0 = time.perf_counter()
        for _ in range(steps):
            assert call() == 0
        dt = time.perf_counter() - t0
        lib.zstdb200_host_free(h_src)
        lib.zstdb200_host_free(h_dst)
        return {"value": round(N * total * steps / dt / 1e9, 3), "unit": "GB/s", "devices": N,
                "what": "one process, one zstdb200 context over all devices, pinned host buffers, verified against the corpus"}
    finally:
        ctx.close()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    g = Gpu(args)
    world = g.world
    w = prepare(args, g.rank)
    if args.dump_outputs and 8 * w["n"] > (12 << 20):
        raise SystemExit(f"--dump-outputs: the result codes of {w['n']} items do not fit the dump's 64 MB; use a larger --chunk")
    decode = w["kind"] == "decode64k"
    if w.get("dictionary"):
        g.ctx.load_dictionary(w["dictionary"])
        args.no_cpu_baseline = True          # the all-core oracle arm has no dictionary entry point
    sampler = ClockSampler(g.local)
    m = measure(g, args, w, args.steps, args.warmup, sampler=sampler, extras=not args.no_extras,
                dump=args.dump_outputs if g.rank == 0 else None)
    sampler.stop_flag = True      # clocks are sampled through both timed regions (device-resident and host-buffer)
    sampler.join()
    n, total, src_bytes, ms, kms = m["n"], m["total"], m["src_bytes"], m["ms"], m["kernel_ms"]
    our_compressed = m["our_compressed"]
    dom = max(kms, key=kms.get)
    algo_bytes = src_bytes + (total if decode else our_compressed)
    peak, peak_src = measured_peak()
    achieved = algo_bytes / (kms[dom] * 1e-3) / 1e9

    # ---------------- the other direction of BASELINE.json's metric (configs[2]): compression at levels 1-3 ----------------
    compress = None
    if decode and args.corpus == "log" and not args.chunk and not args.no_extras and not args.dictionary:
        compress = {}
        for lvl in (1, 2, 3):
            wc = prepare(args, g.rank, workload="compress128k", level=lvl, raw=w["raw"])
            k_steps = max(2, min(args.steps, 3))
            mc = measure(g, args, wc, k_steps, 3)
            cdom = max(mc["kernel_ms"], key=mc["kernel_ms"].get)
            calgo = mc["src_bytes"] + mc["our_compressed"]
            compress[f"L{lvl}"] = {
                "value": round(total * world * k_steps / (mc["ms"] * 1e-3) / 1e9, 3), "unit": "GB/s",
                "e2e": round(total * world * k_steps / mc["e2e_s"] / 1e9, 3),
                "our_ratio": round(total / mc["our_compressed"], 4), "libzstd_ratio": round(total / wc["ref_compressed_bytes"], 4),
                "kernel_ms": {k: round(v, 3) for k, v in mc["kernel_ms"].items()},
                "roofline_frac": round(calgo / (mc["kernel_ms"][cdom] * 1e-3) / 1e9 / peak, 5), "roofline_kernel": cdom,
                "pipeline_frac": round(calgo * k_steps / (mc["ms"] * 1e-3) / 1e9 / peak, 5), "gpu_launches": mc["launches"]}
        compress["workload"] = (f"compress128k: {total} B/GPU of log text in 128 KiB chunks, one frame each with XXH64; ratio comparator = libzstd 1.5.5 at the "
                                "same level (the reference has no compressor: ratio parity is unpinned by the reference)")

    # ---------------- multi-block frames (BASELINE.json configs[4], large end): tick records as 256 KiB and 1 MiB frames ----------------
    multi = None
    if decode and args.corpus == "log" and not args.chunk and not args.no_extras and not args.dictionary and world == 1:
        multi = {}
        for chunk in (262144, 1048576):
            a2 = argparse.Namespace(**vars(args)); a2.corpus = "tick"; a2.chunk = chunk
            wm = prepare(a2, g.rank)
            k_steps = max(2, min(args.steps, 3))
            mm = measure(g, a2, wm, k_steps, 3)
            multi[f"tick_{chunk // 1024}k"] = {
                "value": round(wm["total"] * k_steps / (mm["ms"] * 1e-3) / 1e9, 3), "unit": "GB/s",
                "e2e": round(wm["total"] * k_steps / mm["e2e_s"] / 1e9, 3), "frames": wm["n"], "blocks_per_frame": chunk // 131072,
                "libzstd_ratio": round(wm["total"] / wm["ref_compressed_bytes"], 4),
                "kernel_ms": {k: round(v, 3) for k, v in mm["kernel_ms"].items()}, "gpu_launches": mm["launches"]}
            del wm, mm
        multi["workload"] = (f"decode of {total} B/GPU of libzstd-1.5.5 level-3 tick records held as 256 KiB / 1 MiB frames (2 / 8 blocks each): the "
                             "block-parallel path (DESIGN.md 3b); kernel_ms includes the _blk / _big kernels under their stage's name")

    single = None
    if world > 1 and decode and not args.no_extras:
        g.barrier()
        if g.rank == 0:
            try:
                single = single_context_all_devices(g, args, w, max(1, min(args.steps, 3)))
            except Exception as e:      # e.g. host memory for N x the workload is not available on this box
                single = {"unavailable": str(e)[:200]}
        g.barrier()

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    cpu, cpu_libzstd = None, None
    if g.rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = CpuBaseline(args, w)
        cb.run()
        tt, nb, runs = 0.0, 0, 0
        while tt < 3.0 and runs < 50:
            dt, b = cb.run()
            tt += dt; nb += b; runs += 1
        cpu = {"value": round(nb / tt / 1e9, 3), "unit": "GB/s", "cores": cb.cores, "kind": cb.kind,
               "sample": f"{runs} pass(es) over the full step ({n} frames, {total} B) = {tt * cb.cores:.1f} core-seconds; {cb.what}"}
        cpu_libzstd = libzstd_decode_baseline(cb) if decode else None

    if g.rank == 0:
        steps = args.steps
        value = total * world * steps / (ms * 1e-3) / 1e9
        d2h = (total if decode else our_compressed) + n * 4
        line = {
            "metric": METRIC[args.workload], "value": round(value, 3), "unit": "GB/s", "n_gpus": world,
            "steps": steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms / steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args, w),
            "e2e": {"value": round(total * world * steps / m["e2e_s"] / 1e9, 3), "unit": "GB/s",
                    "h2d_bytes_per_step": int(src_bytes + n * 24), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": m["launches"],
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 5),
                         "traffic": recorded_traffic(f"{args.workload}/{args.corpus}/{w['chunk']}/{total}/L{args.level}", dom), "kernel": dom, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(algo_bytes),
                         "pipeline_frac": round(algo_bytes * steps / (ms * 1e-3) / 1e9 / peak, 5)},
            "kernel_ms": {k: round(v, 4) for k, v in kms.items()},
            "cpu_baseline": cpu,
        }
        if cpu is not None and cpu_libzstd is not None:
            line["cpu_baseline_libzstd"] = cpu_libzstd
        if not decode:
            line["config"]["our_compressed_bytes_per_gpu"] = our_compressed
            line["config"]["our_ratio"] = round(total / our_compressed, 4)
        if "e2e_pageable_s" in m:
            line["e2e_pageable"] = {"contiguous": round(total * world / m["e2e_pageable_s"] / 1e9, 3), "scattered": round(total * world / m["e2e_scattered_s"] / 1e9, 3),
                                    "unit": "GB/s", "what": "the same C-ABI call on pageable (malloc / numpy) caller memory: one array pair, and one array per frame"}
            line["single_call_us"] = round(m["single_call_us"], 1)
        if compress:
            line["compress"] = compress
        if multi:
            line["multi_block"] = multi
        if single:
            line["e2e_single_ctx"] = single
        print(json.dumps(line), flush=True)
    g.ctx.close()
    if g.dist:
        g.dist.destroy_process_group()


if __name__ == "__main__":
    main()
