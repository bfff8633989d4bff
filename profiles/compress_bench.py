"""Compression throughput on the GPU: one JSON line per workload.

Workloads (plaintext of the decode configs): C2b = 8192 x 128 KiB enwik-shaped text (1 GiB), C4 = 4096 x 1 MiB Silesia mix.
Each line: card name and power limit; GB/s of plaintext compressed at the Fastest level with the content checksum, device-resident
input and output, twice: "GBps_call" = CUDA events on the context's stream around >= 10 timed calls of b200z_compress_frames_batch
after warm-up (the call is synchronous: host plan, descriptor upload, results download and stream sync are inside the window), and
"GBps_kernels" = over the sum of the kernels' device time; per-kernel milliseconds (mean of two separate passes under
torch.profiler); the compression ratio, and -- on a fixed, seeded sample of the same frames (--zstd-sample,
default 512) -- libzstd level 1 and level 3 ratios and libzstd level 1 GB/s on all usable host cores (affinity mask capped by the
CPU quota, as bench.py's cpu_baseline).  The plaintexts are generated from the configs' seeds (datagen.config_c2b / config_c4)
without building their compressed frames.  The last timed pass's output is decoded by this library and compared with the input before anything is printed.

    python profiles/compress_bench.py [--workloads c2b,c4] [--steps 10] [--warmup 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True, timeout=30)
        name, power = [x.strip() for x in out.strip().splitlines()[0].split(",")]
        return name, power
    except Exception as e:   # noqa: BLE001
        return f"unknown ({e})", "unknown"


def libzstd_pass(pieces, level, threads):
    import datagen
    with ThreadPoolExecutor(max_workers=threads) as ex:
        return list(ex.map(lambda p: len(datagen.compress(p, level=level, checksum=True)), pieces))


def workload(name):
    """(plaintext, frame offsets, frame sizes) of config C2b / C4 (same generators and seeds as datagen.config_c2b / config_c4)."""
    import datagen
    if name == "c2b":
        plain, frame = datagen.c2_text_plain(1 << 30, 0xE90001), 131072
    elif name == "c4":
        frame = 1 << 20
        with ThreadPoolExecutor(max_workers=datagen.nthreads()) as ex:
            plain = np.concatenate(list(ex.map(lambda i: datagen.gen_silesia_mix(frame, 0xC40000 + i), range(4096))))
    else:
        raise SystemExit(f"unknown workload {name}")
    n = len(plain) // frame
    return plain, np.arange(n, dtype=np.uint64) * frame, np.full(n, frame, dtype=np.uint64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2b,c4")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--zstd-sample", type=int, default=512)
    args = ap.parse_args()
    import torch
    import _pkg
    import bench
    pkg = _pkg.load()
    if not torch.cuda.is_available():
        raise SystemExit("compress_bench.py measures the GPU: no CUDA device")
    ctx = pkg.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream())
    gpu, power = card()
    threads = bench.host_threads()
    for wl in args.workloads.split(","):
        plain, off, size = workload(wl)
        n = len(off)
        d_in = torch.from_numpy(np.ascontiguousarray(plain)).cuda()
        bound = pkg.compress_bound(int(size.max()))
        io = np.zeros(n, dtype=pkg.binding.FRAME_IO_DTYPE)
        io["src_off"], io["src_size"] = off, size
        io["out_off"], io["out_cap"] = np.arange(n, dtype=np.uint64) * bound, bound
        d_out = torch.zeros(n * bound, dtype=torch.uint8, device="cuda")
        for _ in range(args.warmup):
            pkg.compress_frames(ctx, d_in, io, d_out)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms = []
        for _ in range(args.steps):
            ev0.record(stream)
            res = pkg.compress_frames(ctx, d_in, io, d_out)
            ev1.record(stream)
            ev1.synchronize()
            ms.append(ev0.elapsed_time(ev1))
        assert (res["status"] == 0).all()
        # the last timed pass, decoded by this library, must give the input back
        dio = np.zeros(n, dtype=pkg.binding.FRAME_IO_DTYPE)
        dio["src_off"], dio["src_size"], dio["out_off"], dio["out_cap"] = io["out_off"], res["out_size"], off, size
        dec = torch.zeros(len(plain), dtype=torch.uint8, device="cuda")
        dres = pkg.decode_frames(ctx, d_out, dio, dec)
        assert (dres["status"] == 0).all() and torch.equal(dec, d_in), "decoded output differs from the input"
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(2):
                pkg.compress_frames(ctx, d_in, io, d_out)
            torch.cuda.synchronize()
        kernels = {}
        for e in prof.key_averages():
            k = e.key.split("(")[0].split("::")[-1]
            if k in ("k_cxxh64", "k_cmatch", "k_cblock", "k_cframe", "k_cemit"):
                kernels[k] = round(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) / 1000.0 / 2, 3)
        total_in = int(size.sum())
        total_out = int(res["out_size"].sum())
        pick = np.sort(np.random.default_rng(7).choice(n, min(n, args.zstd_sample), replace=False))
        pieces = [plain[int(off[i]):int(off[i] + size[i])] for i in pick]
        sample_in = sum(len(p) for p in pieces)
        sample_ours = int(res["out_size"][pick].sum())
        t0 = time.perf_counter()
        z1 = sum(libzstd_pass(pieces, 1, threads))
        t1 = time.perf_counter()
        z3 = sum(libzstd_pass(pieces, 3, threads))
        med = float(np.median(ms))
        print(json.dumps({
            "workload": wl, "frames": n, "plaintext_bytes": total_in, "gpu": gpu, "power_limit": power, "level": "fastest", "checksum": True,
            "GBps_call": round(total_in / (med * 1e-3) / 1e9, 2), "GBps_kernels": round(total_in / (sum(kernels.values()) * 1e-3) / 1e9, 2),
            "ms_median": round(med, 3), "ms_min": round(min(ms), 3), "ms_max": round(max(ms), 3),
            "timed_passes": args.steps, "kernel_ms": kernels,
            "ratio": round(total_in / total_out, 4), "zstd_sample_frames": len(pick), "ratio_on_sample": round(sample_in / sample_ours, 4),
            "libzstd_l1_ratio": round(sample_in / z1, 4), "libzstd_l3_ratio": round(sample_in / z3, 4),
            "libzstd_l1_GBps_host": round(sample_in / (t1 - t0) / 1e9, 2), "host_threads": threads,
            "blocks": {"raw": int(res["raw_blocks"].sum()), "rle": int(res["rle_blocks"].sum()), "compressed": int(res["compressed_blocks"].sum())},
        }), flush=True)
        del d_in, d_out, dec
        torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
