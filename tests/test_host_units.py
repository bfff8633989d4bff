"""Host-compiled unit checks of device/host shared code (no GPU needed: nvcc compiles the __host__ __device__ helpers for the host)."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="nvcc not available")
def test_description_bit_readers_match_bit_serial_reference(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = str(tmp_path / "bit_readers_test")
    subprocess.check_call([nvcc, "-x", "cu", "-std=c++17", "-O2", "-w", "-o", exe, os.path.join(HERE, "host", "bit_readers_test.cpp")])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stdout + out.stderr


def test_bench_reference_arm_line(tmp_path):
    """`bench.py --impl reference` (the restated CPU path on the host cores) prints the contract's JSON line on a small workload."""
    import json
    root = os.path.dirname(HERE)
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--frames", "64", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "decompressed_GBps" and line["unit"] == "GB/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def _bench_dump(tmp_path, *args):
    """Runs bench.py with --dump-outputs on a 64-frame C2b workload; checks the dumped sample against the generator's
    plaintext and returns the arrays."""
    import datagen
    root = os.path.dirname(HERE)
    d = tmp_path / "outputs"
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), *args, "--frames", "64", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    a = {f[:-len(".npy")]: np.load(d / f) for f in os.listdir(d)}
    assert all(v.dtype in (np.float32, np.float64) for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20
    fs = datagen.config_c2b(total_bytes=64 * 131072, frame_bytes=131072)
    idx, fi = a["output_index"].astype(np.int64), a["frame_index"].astype(np.int64)
    assert len(idx) == len(a["output"]) > 0 and np.array_equal(a["output"], fs.plain[idx])
    assert np.array_equal(fi, np.arange(fs.nframes)) and np.array_equal(a["frame_out_size"], fs.out_size)
    return a, fs


def test_bench_dump_outputs_reference_arm(tmp_path):
    _bench_dump(tmp_path, "--impl", "reference")


@pytest.mark.gpu
def test_bench_dump_outputs(tmp_path, oracle):
    a, fs = _bench_dump(tmp_path, "--skip-cpu", "--e2e-steps", "1")
    assert (a["frame_status"] == 0).all() and np.array_equal(a["frame_bytes_read"], fs.src_size)
    plain = [fs.plain[int(o):int(o + n)] for o, n in zip(fs.out_off, fs.out_size)]
    assert np.array_equal(a["frame_calculated_checksum"], [oracle.xxh64(p) & 0xFFFFFFFF for p in plain])
