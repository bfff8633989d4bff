#!/usr/bin/env python3
"""bench.py -- decompressed GB/s of the zstd block-decompression hot path on enwik9-shaped frames (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (restated port) on host cores
    python bench.py --config c2a|c3|c4|c5                    # the other BASELINE.json configs at their full sizes

A "step" is one pass of the hot path over the whole workload: config C2b = enwik9-shaped text, 8192 independent
128 KiB single-block frames (1 GiB), level 3, checksums on.  `value` is measured with compressed frames, block
descriptors and output all resident in HBM (kernel launches only inside the timed region, the content checksum of every
frame included, as the reference computes it); `e2e` is the same work through the C-ABI one-shot call with HOST buffers
(host planning + H2D + kernels + D2H inside the timed region).
Multi-GPU: frames are independent, no data-path collective (NCCL only gathers the timings).  Both scalings are measured
in one run: weak (every rank decodes the whole workload) and strong (the frames are sharded across the ranks,
SURVEY 8(e)); --scaling picks which one is `value`, the other is reported under `<mode>_scaling`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GB = 1e9


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region, in-process through NVML (nvidia_ml_py).  A polling
    `nvidia-smi -lms` child per rank stalls kernel submission on multi-GPU boxes (measured: 4.4 -> 220 ms per step at N=2),
    so it is only the fallback when NVML cannot be loaded."""

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread, self.stop_flag = index, [], None, None, False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def _poll_nvml(self):
        N = self.nvml
        bits = {"hw_slowdown": getattr(N, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_thermal_slowdown": getattr(N, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(N, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_power_cap": getattr(N, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(N, "nvmlDeviceGetCurrentClocksThrottleReasons")
        mx = N.nvmlDeviceGetMaxClockInfo(self.handle, N.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                sm = N.nvmlDeviceGetClockInfo(self.handle, N.NVML_CLOCK_SM)
                r = int(get_reasons(self.handle))
                self.rows.append([str(sm), str(mx), "0"] + ["Active" if r & bits[k] else "Not Active" for k in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")])
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "250", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


WORKLOADS = {
    # name: (BASELINE.json config, builder(args), description)
    "c2b": "C2b enwik9-shaped text, {n} independent {fb}-byte single-block frames, level 3, checksum on",
    "c2a": "C2a enwik9-shaped text as {n} frame(s) of chained 128 KiB blocks (windowLog 17), level 3, checksum on",
    "c3": "C3 {n} independent 64 KiB frames, 4-stream-Huffman-heavy literals, level 3",
    "c4": "C4 Silesia-mix-shaped, {n} frames of 1 MiB (8 chained blocks, RLE / raw / compressed), level 3",
    "c5": "C5 {n} small frames sharing one 110 KiB raw-content dictionary, level 3",
}


def build_workload(args):
    import datagen as G
    c = args.config
    if c == "c2b":
        return G.config_c2b(total_bytes=args.frames * args.frame_bytes, frame_bytes=args.frame_bytes)
    if c == "c2a":
        return G.config_c2a(total_bytes=args.c2a_bytes, nframes=args.c2a_frames)
    if c == "c3":
        return G.config_c3(nframes=args.c3_frames)
    if c == "c4":
        return G.config_c4(nframes=args.c4_frames)
    if c == "c5":
        return G.config_c5(nframes=args.c5_frames)
    raise SystemExit("unknown --config " + c)


def load_workload(args, rank, barrier):
    if rank == 0:
        fs = build_workload(args)   # rank 0 fills the on-disk cache, the others read it
    barrier()
    if rank != 0:
        fs = build_workload(args)
    return fs


def workload_config(args, fs):
    """The `config` object both arms print (same workload, same keys)."""
    return {"workload": WORKLOADS[args.config].format(n=fs.nframes, fb=args.frame_bytes), "config": args.config,
            "frames": fs.nframes, "D_bytes": fs.D, "C_bytes": fs.C, "ratio": fs.D / max(fs.C, 1), "sha256_plain": fs.sha256()[:16],
            "content_checksum_computed": True,
            "l2": "inputs larger than L2 (C+D per pass = %.0f MB vs 126 MB L2)" % ((fs.C + fs.D) / 1e6),
            "parallelism": "frames are independent: one process per GPU, no data-path collective"}


def host_threads():
    """Threads the CPU arm may really use: the affinity mask, capped by the container's CPU quota (cgroup cpu.max /
    cfs_quota) -- more runnable threads than quota only buys throttling (round 1: 2.4 vs 13 GB/s on two boxes)."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        n = max(1, os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.999)))
    return n


def bind_near_gpu(index):
    """Pin this process (and the pinned host buffers it allocates afterwards) to the CPUs next to GPU `index`: on an 8-GPU box
    the ranks otherwise share one socket's memory controllers and the PCIe copies of GPUs 4-7 cross the inter-socket link."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/local_cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-"); cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"gpu": index, "pci": bus, "cpus": len(cpus)}
    except Exception as e:
        return {"gpu": index, "error": str(e)[:80]}
    return {"gpu": index, "cpus": 0}


def cpu_decode_pass(fs, threads, buf=None):
    """One pass of the reference's CPU path (restated port) over ALL frames of the workload, one FrameDecoder per thread."""
    from oracle import oracle as O
    rd = fs.raw_dict.tobytes() if fs.raw_dict is not None else None
    if buf is None:
        buf = np.zeros(fs.D + 64, dtype=np.uint8)   # pre-touched: page faults stay out of the timing
    t0 = time.perf_counter()
    out, sizes = O.bulk_decode(fs.comp, fs.src_off, fs.src_size, fs.out_off, fs.out_size, raw_dict=rd, nthreads=threads, out=buf)
    return time.perf_counter() - t0, out, sizes


def libzstd_one_core(fs, budget_s=2.0):
    """libzstd 1.5.5 (system library), one thread, on the first frames of the workload: the anchor for the reference README's
    'ruzstd is 1.4-3.5x slower than zstd' (Readme.md:25-29)."""
    import datagen as G
    rd = fs.raw_dict.tobytes() if fs.raw_dict is not None else None
    done, t0 = 0, time.perf_counter()
    for i in range(fs.nframes):
        f = fs.comp[int(fs.src_off[i]):int(fs.src_off[i] + fs.src_size[i])]
        G.decompress(f, int(fs.out_size[i]), raw_dict=rd)
        done += int(fs.out_size[i])
        if time.perf_counter() - t0 > budget_s:
            break
    return done / (time.perf_counter() - t0) / GB


def cpu_baseline(fs, threads=None, passes=2):
    """The restated CPU path (oracle 'port' of ruzstd's FrameDecoder loop) on the host cores: every frame of the workload,
    all the threads this process may use."""
    from oracle import oracle as O
    threads = threads or host_threads()
    k = min(fs.nframes, 64)
    sub = fs.subset(0, k)
    cpu_decode_pass(sub, 1)
    one = min(cpu_decode_pass(sub, 1)[0] for _ in range(2))
    buf = np.zeros(fs.D + 64, dtype=np.uint8)
    cpu_decode_pass(fs, threads, buf)   # warm-up (page tables, thread stacks)
    best, out = None, None
    for _ in range(passes):
        dt, out, _ = cpu_decode_pass(fs, threads, buf)
        best = dt if best is None else min(best, dt)
    assert np.array_equal(out[:fs.D], fs.plain), "CPU port output differs from the generator's plaintext"
    return {"value": fs.D / best / GB, "unit": "GB/s", "cores": threads, "kind": "port",
            "sample": f"all {fs.nframes} frames ({fs.D / 2**20:.0f} MiB) of the same workload, one FrameDecoder per thread, best of {passes} passes after a warm-up",
            "one_core_GBps": sub.D / one / GB, "libzstd_1.5.5_one_core_GBps": libzstd_one_core(fs)}


DUMP_BYTES = 1 << 21    # --dump-outputs: decoded bytes kept (float32 value + float64 position: 24 MiB)
DUMP_FRAMES = 1 << 19   # and frames kept (five float64 arrays: at most 20 MiB)


def sample_index(n, cap):
    """Sorted positions of a fixed, seeded sample of `cap` of `n` items (all of them when n <= cap)."""
    if n <= cap:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.Generator(np.random.PCG64(0xD0D0)).choice(n, cap, replace=False, shuffle=False))


def dump_outputs(path, out_index, out_values, frames):
    """--dump-outputs: write what the timed path returned in its last step as float32 / float64 .npy files, so that two builds
    run with the same arguments can be compared output for output.  output.npy holds the decoded bytes at the positions in
    output_index.npy (offsets into the concatenated output of all frames); frame_<field>.npy holds the per-frame results
    {field: array over all frames} of the frames listed in frame_index.npy."""
    os.makedirs(path, exist_ok=True)
    fi = sample_index(len(next(iter(frames.values()))), DUMP_FRAMES)
    arrays = {"output_index": out_index.astype(np.float64), "output": np.asarray(out_values).astype(np.float32), "frame_index": fi.astype(np.float64)}
    arrays.update({"frame_" + k: np.asarray(v)[fi].astype(np.float64) for k, v in frames.items()})
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (restated port; ruzstd is Rust and cannot be
    built in this image) on the host cores, same workload / config / metric; each step = one pass over every frame."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    fs = load_workload(args, 0, lambda: None)
    threads = host_threads()
    buf = np.zeros(fs.D + 64, dtype=np.uint8)
    steps = max(1, args.steps if args.steps_given else 5)
    warm = max(1, min(args.warmup, 3))
    times = []
    for i in range(warm + steps):
        dt, out, sizes = cpu_decode_pass(fs, threads, buf)
        if i >= warm:
            times.append(dt)
    assert np.array_equal(out[:fs.D], fs.plain), "CPU port output differs from the generator's plaintext"
    if args.dump_outputs:
        bi = sample_index(fs.D, DUMP_BYTES)
        dump_outputs(args.dump_outputs, bi, out[bi], {"out_size": sizes})
    dt = sum(times)
    val = fs.D * steps / dt / GB
    line = {"impl": "reference", "metric": "decompressed_GBps", "value": val, "unit": "GB/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": dt / steps * 1e3, "ms_per_step_min": min(times) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": workload_config(args, fs), "bit_exact": True,
            "cpu_baseline": {"value": val, "unit": "GB/s", "cores": threads, "kind": "port",
                             "sample": f"all {fs.nframes} frames ({fs.D / 2**20:.0f} MiB) per step, one FrameDecoder per thread (content checksum computed, like FrameDecoder)",
                             "libzstd_1.5.5_one_core_GBps": libzstd_one_core(fs)},
            "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def time_passes(batch, d_out, stream, steps, barrier, torch):
    """K passes of the device-resident path, CUDA events on the library's stream, barrier + synchronize on both sides."""
    barrier(); torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        batch.run(d_out)
    ev1.record(stream)
    stream.synchronize(); torch.cuda.synchronize(); barrier()
    return ev0.elapsed_time(ev1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="c2b", choices=sorted(WORKLOADS), help="BASELINE.json config; c2b is the one the metric is quoted on")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = every rank decodes the whole workload; strong = the frames are sharded across ranks (SURVEY 8(e)). "
                         "The other one is measured too and reported under its own key.")
    ap.add_argument("--frames", type=int, default=8192)
    ap.add_argument("--frame-bytes", type=int, default=131072)
    ap.add_argument("--c2a-bytes", type=int, default=1 << 30)
    ap.add_argument("--c2a-frames", type=int, default=1)
    ap.add_argument("--c3-frames", type=int, default=10000)
    ap.add_argument("--c4-frames", type=int, default=4096)
    ap.add_argument("--c5-frames", type=int, default=100000)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                    "(a seeded sample of the decoded bytes and the per-frame results; with N > 1, those of rank 0)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    args.steps_given = args.steps is not None
    if args.steps is None:
        args.steps = 50 if args.config != "c2a" else 3   # one chained 1 GiB frame is a serial chain of 8192 blocks: seconds per pass
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    numa = bind_near_gpu(local) if world > 1 else None   # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)

    def max_over_ranks(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if world == 1:
            return [float(x)]
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        return [float(v.item()) for v in allt]

    import _pkg
    pkg = _pkg.load()
    from importlib import import_module
    sharding = import_module("zstd_rs_b200.sharding")
    fs_all = load_workload(args, rank, barrier)
    ctx = pkg.Context(local)
    ctx.set_flags(pkg.binding.FLAG_CHECKSUM)   # the reference hashes every frame it drains (decode_buffer.rs:225-226): so does the timed pass
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local))
    dic = pkg.Dictionary.raw_content(ctx, 1, fs_all.raw_dict.tobytes()) if fs_all.raw_dict is not None else None

    def measure(fs, label):
        """device-resident passes + end-to-end calls on frame set `fs` of this rank"""
        io = fs.frames_io()
        D = fs.D
        batch = pkg.Batch(ctx, fs.comp, io, forced_dict=dic)
        d_out = torch.empty(D + 64, dtype=torch.uint8, device="cuda")
        for _ in range(args.warmup):
            batch.run(d_out)
        stream.synchronize()
        res = batch.finish()
        assert (res["status"] == 0).all(), (label, res[res["status"] != 0][:3])
        assert (res["calculated_checksum"] == res["checksum_from_data"])[res["has_checksum"] == 1].all(), "content checksum mismatch"
        got = d_out[:D].cpu().numpy()
        bit_exact = bool(np.array_equal(got, fs.plain))
        assert bit_exact, label + ": GPU output differs from the generator's plaintext"
        del got
        sampler = ClockSampler(local)
        sampler.start()
        t_wait = time.time()
        while not sampler.rows and time.time() - t_wait < 5.0:   # the sampler needs a moment before its first sample
            batch.run(d_out); stream.synchronize()
        sampler.rows.clear()
        launches0 = ctx.kernel_launches()
        ms = time_passes(batch, d_out, stream, args.steps, barrier, torch)
        clocks = sampler.stop()
        launches = ctx.kernel_launches() - launches0
        res = batch.finish()
        assert (res["status"] == 0).all(), "a frame failed inside the timed region: %r" % (res[res["status"] != 0][:3],)
        last = None
        if args.dump_outputs:   # what the last timed pass left in d_out, before any later pass reuses it
            bi = sample_index(D, DUMP_BYTES)
            last = (bi, d_out[torch.from_numpy(bi).to(d_out.device)].cpu().numpy(),
                    {k: res[k] for k in ("status", "out_size", "bytes_read", "calculated_checksum")})
        out = {"last_step": last, "fs": fs, "batch": batch, "d_out": d_out, "bit_exact": bit_exact, "ms": ms, "launches": launches, "clocks": clocks, "info": batch.info(),
               "sched": batch.debug_sched()}
        # the same passes without the checksum stage (what round 1 timed)
        ctx.set_flags(0)
        batch.run(d_out); stream.synchronize()
        out["ms_nochk"] = time_passes(batch, d_out, stream, max(3, args.steps // 5), barrier, torch) / max(3, args.steps // 5)
        ctx.set_flags(pkg.binding.FLAG_CHECKSUM)
        return out

    def measure_e2e(fs):
        """the public one-shot call with pinned HOST buffers: plan + H2D + kernels + D2H inside the timed region"""
        if args.e2e_steps <= 0:
            return float("nan")
        h_in = torch.from_numpy(np.ascontiguousarray(fs.comp)).pin_memory()
        h_out = torch.empty(fs.D + 64, dtype=torch.uint8).pin_memory()
        io = fs.frames_io()
        ts = []
        for i in range(1 + args.e2e_steps):
            barrier(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = pkg.decode_frames(ctx, h_in, io, h_out, forced_dict=dic)
            dt = (time.perf_counter() - t0) * 1e3
            assert (r["status"] == 0).all()
            if i > 0:
                ts.append(dt)
        assert np.array_equal(h_out[:fs.D].numpy(), fs.plain), "e2e output differs"
        return float(np.mean(ts))

    # ---- weak: every rank decodes the whole workload.  strong: contiguous shards balanced by compressed bytes (sharding.py)
    lo, hi = sharding.shard_frames(fs_all.src_size, world, rank) if world > 1 else (0, fs_all.nframes)
    fs_shard = fs_all.subset(lo, hi) if world > 1 else fs_all
    runs = {}
    order = ["weak", "strong"] if world > 1 else ["weak"]
    for mode in order:
        fs = fs_all if mode == "weak" else fs_shard
        m = measure(fs, mode)
        m["ms_max"] = max_over_ranks(m["ms"])
        m["ms_per_rank"] = [x / args.steps for x in all_ranks(m["ms"])]
        m["e2e_ms"] = max_over_ranks(measure_e2e(fs))
        m["D_total"] = fs_all.D * world if mode == "weak" else fs_all.D
        m["C_total"] = fs_all.C * world if mode == "weak" else fs_all.C
        runs[mode] = m
    main_mode = args.scaling if world > 1 else "weak"
    M = runs[main_mode]
    fs, batch, d_out = M["fs"], M["batch"], M["d_out"]
    ms_per_step = M["ms_max"] / args.steps
    value = M["D_total"] / (ms_per_step * 1e-3) / GB

    # ---- per-kernel durations, live (CUDA events between the kernels on the launching stream)
    if d_out is None:
        d_out = torch.empty(fs.D + 64, dtype=torch.uint8, device="cuda")
    prof = [batch.run_profile(d_out) for _ in range(5)]
    kern_ms = {k: float(np.median([p[k] for p in prof])) for k in prof[0]}
    tot = sum(kern_ms.values())
    timeline = {k: v for k, v in batch.run_timeline(d_out).items() if v >= 0}
    dominant = max(kern_ms, key=kern_ms.get)

    if rank == 0:
        peak, peak_src = measured_peak()
        # roofline of THIS rank's pass (per-GPU quantity): algorithmic bytes of the rank's frames over the rank's pass time
        achieved = (fs.C + fs.D) / (M["ms"] / args.steps * 1e-3) / GB
        traffic = None   # ncu DRAM bytes of one pass: captured for the C2b workload on one GPU only (profiles/traffic.py)
        if args.config == "c2b" and fs.nframes == 8192:
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("pipeline_dram_bytes_per_step")
            except Exception:
                pass
        cfg = workload_config(args, fs_all)   # identical in both arms
        run = {"frames_per_gpu": fs.nframes, "D_bytes_per_gpu": fs.D, "C_bytes_per_gpu": fs.C, "blocks_per_gpu": M["info"]["blocks"],
               "sequences_per_gpu": M["info"]["sequences"],
               "ranks": (f"{world} ranks, every rank decodes the whole workload" if main_mode == "weak" else f"{world} ranks, frames sharded contiguously by compressed bytes"),
               "exec_kernels": M["sched"]}
        line = {
            "metric": "decompressed_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "ms_per_step_per_rank": M["ms_per_rank"], "higher_is_better": True, "scaling": main_mode, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": cfg, "run": run,
            "bit_exact": M["bit_exact"],
            "gpu_launches": int(M["launches"]),
            "clocks": M["clocks"],
            "value_without_checksum_stage": M["D_total"] / (max_over_ranks(M["ms_nochk"]) * 1e-3) / GB if world == 1 else None,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "algorithmic_bytes_per_step": fs.C + fs.D,
                         "kernel": "whole pass (k_setup, k_huf || k_fse, k_exec_cta / k_exec, k_xxh64), CUDA events over the timed region on the library stream",
                         "dominant_kernel": dominant, "kernel_ms": kern_ms, "completion_ms": timeline, "kernel_share": {k: v / tot for k, v in kern_ms.items()},
                         "read_only_GBps": fs.C / (M["ms"] / args.steps * 1e-3) / GB},
            "e2e": {"value": M["D_total"] / (M["e2e_ms"] * 1e-3) / GB, "unit": "GB/s", "h2d_bytes_per_step": int(fs.C), "d2h_bytes_per_step": int(fs.D), "ms_per_step": M["e2e_ms"],
                    "steps": args.e2e_steps, "call": "b200z_decode_frames_batch with pinned host input/output"},
        }
        for mode, m in runs.items():
            if mode != main_mode:
                line[mode + "_scaling"] = {"value": m["D_total"] / (m["ms_max"] / args.steps * 1e-3) / GB, "unit": "GB/s", "ms_per_step": m["ms_max"] / args.steps,
                                           "ms_per_step_per_rank": m["ms_per_rank"], "frames_per_gpu": m["fs"].nframes, "bit_exact": m["bit_exact"],
                                           "e2e": {"value": m["D_total"] / (m["e2e_ms"] * 1e-3) / GB, "unit": "GB/s", "ms_per_step": m["e2e_ms"]}}
        if numa is not None:
            line["cpu_affinity"] = numa
        if not args.skip_cpu and world == 1:   # the CPU baseline is a single-GPU-run companion (rank 0, N = 1 only)
            line["cpu_baseline"] = cpu_baseline(fs_all)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *M["last_step"])
        print(json.dumps(line))
    barrier()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
