"""Compression (b200z_compress_frames_batch / b200z_compress; ruzstd's encoding::{compress, compress_to_vec, FrameCompressor} at
the Uncompressed and Fastest levels).

CPU: the encoder pieces of csrc/enc.cuh compiled for the host and checked against the decoder's parsers in tables.cuh, and a
whole-frame rehearsal through the same block and frame writers decoded by the oracle and by libzstd; ABI facts.
GPU: every frame decodes to its input with libzstd, the oracle (ruzstd's decoding semantics) and this library in both
execution modes; header facts, byte identity of the Uncompressed level, block-type decisions, determinism, ratio gates."""
import hashlib
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, read_golden

HERE = os.path.dirname(os.path.abspath(__file__))
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
BLOCK = 131072


@pytest.fixture(scope="module")
def encoder_exe(tmp_path_factory):
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("enc") / "encoder_test")
    subprocess.check_call([NVCC, "-x", "cu", "-std=c++17", "-O2", "-w", "-o", exe, os.path.join(HERE, "host", "encoder_test.cpp")])
    return exe


def corpus_plaintexts(oracle, manifest):
    """The reference's encode corpus (encode_corpus.rs): the plaintexts of the decodecorpus frames, checked by SHA-256."""
    out = {}
    for name in sorted(os.listdir(os.path.join(GOLDEN, "decodecorpus"))):
        plain = oracle.decode_frame(read_golden("decodecorpus", name))[0]
        assert hashlib.sha256(plain).hexdigest() == manifest["corpus"][name]["sha256"], name
        out[name] = plain
    return out


def sample_inputs():
    import datagen
    rng = np.random.default_rng(20261017)
    return {
        "text": bytes(datagen.gen_text(300000, 11)),
        "silesia_mix": bytes(datagen.gen_silesia_mix(400000, 12)),
        "skewed": bytes(datagen.gen_skewed_bytes(200000, 13)),
        "records": bytes(datagen.gen_binary_records(200000, 14)),
        "empty": b"",
        "one": b"Z",
        "five": b"abcab",
        "all_equal": b"\x07" * 300000,
        "block_exact": bytes(datagen.gen_text(BLOCK, 15)),
        "block_plus_1": bytes(datagen.gen_text(BLOCK + 1, 16)),
        "random": rng.integers(0, 256, 250000, dtype=np.uint8).tobytes(),
        "all_256": bytes(range(256)) * 700,
        "long_runs": bytes(np.repeat(rng.integers(0, 4, 3000, dtype=np.uint8), rng.integers(1, 300, 3000)).tobytes()),
    }


# ---------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------
def test_encoder_units_against_decoder_parsers(encoder_exe):
    out = subprocess.run([encoder_exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stdout + out.stderr


def test_whole_frame_rehearsal_decodes_with_oracle_and_libzstd(encoder_exe, oracle, manifest, tmp_path):
    import datagen
    inputs = dict(sample_inputs())
    for name, plain in corpus_plaintexts(oracle, manifest).items():
        inputs["corpus/" + name] = plain
    for name, plain in inputs.items():
        src, dst = tmp_path / "in.bin", tmp_path / "out.zst"
        src.write_bytes(plain)
        subprocess.check_call([encoder_exe, "frame", str(src), str(dst)])
        frame = dst.read_bytes()
        assert oracle.decode_frame(frame)[0] == plain, name
        assert datagen.decompress(frame, len(plain) + 1) == plain, name


def test_compress_result_layout_and_bound(pkg, tmp_path):
    B = pkg.binding
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "b200zstd.h"', 'int main(void) {',
             '  printf("* %zu\\n", sizeof(b200z_compress_result));']
    lines += [f'  printf("{f} %zu %zu\\n", offsetof(b200z_compress_result, {f}), sizeof(((b200z_compress_result *)0)->{f}));'
              for f in B.COMPRESS_RESULT_DTYPE.names]
    lines += ['  return 0;', '}']
    (tmp_path / "l.c").write_text("\n".join(lines))
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(tmp_path / "l.c"), "-o", str(tmp_path / "l")])
    for ln in subprocess.check_output([str(tmp_path / "l")]).decode().split("\n"):
        if ln:
            f, a, *b = ln.split()
            if f == "*":
                assert int(a) == B.COMPRESS_RESULT_DTYPE.itemsize
            else:
                assert B.COMPRESS_RESULT_DTYPE.fields[f][1] == int(a) and B.COMPRESS_RESULT_DTYPE.fields[f][0].itemsize == int(b[0]), f
    # header 6 + Frame_Content_Size field + 3 per block (an input that fills its last block gets an empty one) + data + checksum
    for n, fcs in [(0, 4), (1, 4), (255, 4), (256, 2), (65535, 2), (65536, 4), (BLOCK, 4), (BLOCK + 1, 4), (1 << 32, 8)]:
        assert pkg.compress_bound(n) == 6 + fcs + 3 * (n // BLOCK + 1) + n + 4, n


def test_unimplemented_levels_are_refused_without_a_device(pkg):
    L = pkg.lib()
    for level in (pkg.LEVEL_DEFAULT, pkg.LEVEL_BETTER, pkg.LEVEL_BEST):
        assert L.b200z_compress_frames_batch(None, None, 0, 0, None, 0, level, 0, None, 0, 0, None) == pkg.binding.ERR_REFERENCE_WOULD_PANIC
        assert L.b200z_compress(None, pkg.binding.READ_FN(0), None, pkg.binding.WRITE_FN(0), None, level, 0) == pkg.binding.ERR_REFERENCE_WOULD_PANIC
        with pytest.raises(pkg.B200ZError) as e:
            pkg.compress(None, b"abc", level=level)
        assert e.value.code == pkg.binding.ERR_REFERENCE_WOULD_PANIC
    assert L.b200z_compress_frames_batch(None, None, 0, 0, None, 0, 7, 0, None, 0, 0, None) == 220   # INVALID_ARGUMENT
    assert L.b200z_compress_frames_batch(None, None, 0, 0, None, 0, 1, 0, None, 0, 0, None) == 220   # no context


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
def ruzstd_uncompressed_frame(plain, checksum, xxh64):
    """FrameHeader::serialize + BlockHeader::serialize as FrameCompressor::compress writes them at CompressionLevel::Uncompressed."""
    out = bytearray(b"\x28\xb5\x2f\xfd")
    out.append(4 if checksum else 0)
    out.append(7 << 3)
    pos = 0
    while True:
        chunk = plain[pos:pos + BLOCK]
        pos += len(chunk)
        last = len(chunk) < BLOCK
        out += ((len(chunk) << 3) | int(last)).to_bytes(3, "little")
        out += chunk
        if last:
            break
    if checksum:
        out += (xxh64(plain) & 0xFFFFFFFF).to_bytes(4, "little")
    return bytes(out)


def batch(pkg, ctx, plains, level, checksum=True, content_size=False, device=False, out_caps=None):
    import torch
    src = b"".join(plains)
    caps = out_caps or [pkg.compress_bound(len(p)) for p in plains]
    io = np.zeros(len(plains), dtype=pkg.binding.FRAME_IO_DTYPE)
    so = oo = 0
    for i, p in enumerate(plains):
        io[i] = (so, len(p), oo, caps[i])
        so += len(p)
        oo += caps[i]
    if device:
        inp = torch.frombuffer(bytearray(src) or bytearray(1), dtype=torch.uint8).cuda()[:len(src)]
        out = torch.zeros(max(oo, 1), dtype=torch.uint8, device="cuda")
    else:
        inp, out = src, np.zeros(max(oo, 1), dtype=np.uint8)
    res = pkg.compress_frames(ctx, inp, io, out, level=level, checksum=checksum, content_size=content_size)
    host = out.cpu().numpy() if device else out
    frames = [host[int(io[i]["out_off"]):int(io[i]["out_off"]) + int(res[i]["out_size"])].tobytes() for i in range(len(plains))]
    return frames, res


def decode_with_library(pkg, ctx, frames, sizes, mode):
    old = os.environ.get("B200Z_EXEC_MODE")
    os.environ["B200Z_EXEC_MODE"] = mode
    try:
        comp = b"".join(frames)
        io = np.zeros(len(frames), dtype=pkg.binding.FRAME_IO_DTYPE)
        so = oo = 0
        for i, (f, n) in enumerate(zip(frames, sizes)):
            io[i] = (so, len(f), oo, n)
            so += len(f)
            oo += n
        out = np.zeros(oo + 16, dtype=np.uint8)
        res = pkg.decode_frames(ctx, comp, io, out)
        return [out[int(io[i]["out_off"]):int(io[i]["out_off"]) + int(res[i]["out_size"])].tobytes() if res[i]["status"] == 0 else None
                for i in range(len(frames))], res
    finally:
        if old is None:
            os.environ.pop("B200Z_EXEC_MODE", None)
        else:
            os.environ["B200Z_EXEC_MODE"] = old


@pytest.mark.gpu
@pytest.mark.parametrize("level", [0, 1])
@pytest.mark.parametrize("flags", [0, 1, 2, 3])
def test_round_trip_three_decoders(pkg, ctx, oracle, manifest, level, flags):
    import datagen
    inputs = sample_inputs()
    inputs.update({"corpus/" + k: v for k, v in corpus_plaintexts(oracle, manifest).items()})
    if level == 1 and flags == 3:
        inputs["multi_16mib"] = bytes(datagen.gen_silesia_mix(16 << 20, 17))
    names, plains = list(inputs), list(inputs.values())
    frames, res = batch(pkg, ctx, plains, level, checksum=bool(flags & 1), content_size=bool(flags & 2), device=(flags == 3))
    assert (res["status"] == 0).all()
    for name, p, f, r in zip(names, plains, frames, res):
        assert r["num_blocks"] == len(p) // BLOCK + 1 and len(f) <= pkg.compress_bound(len(p)), name
        assert datagen.decompress(f, len(p) + 1) == p, name
        got, d = oracle.decode_frame(f)
        assert got == p, name
        if flags & 1:
            assert int.from_bytes(f[-4:], "little") == (pkg.xxh64(p) & 0xFFFFFFFF) == r["checksum"], name
            assert d.get_checksum_from_data() == r["checksum"], name
        if flags & 2:
            assert d.content_size() == len(p), name
    for mode in ("warp", "cta"):
        got, dres = decode_with_library(pkg, ctx, frames, [len(p) for p in plains], mode)
        for name, p, g in zip(names, plains, got):
            assert g == p, (mode, name)


@pytest.mark.gpu
def test_decodes_with_a_128k_window_limit(pkg, ctx):
    import datagen
    p = bytes(datagen.gen_text(1 << 20, 21))
    f = pkg.compress(ctx, p)
    d = pkg.FrameDecoder(ctx)
    d.set_max_window_size(BLOCK)
    assert d.decode_all(f, len(p)) == p


@pytest.mark.gpu
@pytest.mark.parametrize("checksum", [False, True])
def test_uncompressed_is_byte_identical_to_the_reference(pkg, ctx, checksum):
    plains = list(sample_inputs().values())
    frames, res = batch(pkg, ctx, plains, pkg.LEVEL_UNCOMPRESSED, checksum=checksum)
    for p, f in zip(plains, frames):
        assert f == ruzstd_uncompressed_frame(p, checksum, pkg.xxh64)
    assert pkg.compress(ctx, plains[0], level=pkg.LEVEL_UNCOMPRESSED, checksum=checksum) == frames[0]


@pytest.mark.gpu
def test_block_type_decisions(pkg, ctx):
    s = sample_inputs()
    frames, res = batch(pkg, ctx, [s["all_equal"], s["random"], s["text"]], pkg.LEVEL_FASTEST, content_size=True)
    eq, rnd, txt = res
    assert eq["rle_blocks"] == eq["num_blocks"] and eq["raw_blocks"] == 0 and eq["compressed_blocks"] == 0
    assert rnd["raw_blocks"] == rnd["num_blocks"] and rnd["out_size"] == pkg.compress_bound(len(s["random"]))
    # text: every non-empty block is Compressed (300000 bytes: 3 blocks)
    assert txt["compressed_blocks"] == txt["num_blocks"] == 3


@pytest.mark.gpu
def test_deterministic_across_batches(pkg, ctx):
    import datagen
    plains = [bytes(datagen.gen_silesia_mix(200000 + 5000 * i, 30 + i)) for i in range(12)]
    a, _ = batch(pkg, ctx, plains, pkg.LEVEL_FASTEST)
    b, _ = batch(pkg, ctx, plains, pkg.LEVEL_FASTEST, device=True)
    assert a == b
    order = np.random.default_rng(5).permutation(len(plains))
    extra = [bytes(datagen.gen_text(70000, 99))]
    c, _ = batch(pkg, ctx, extra + [plains[i] for i in order], pkg.LEVEL_FASTEST)
    assert [c[1 + list(order).index(i)] for i in range(len(plains))] == a


@pytest.mark.gpu
@pytest.mark.parametrize("kind,gate", [("text", 1.15), ("silesia_mix", 1.40), ("skewed", 1.10)])
def test_ratio_gates_against_libzstd_level1(pkg, ctx, kind, gate):
    import datagen
    gen = {"text": datagen.gen_text, "silesia_mix": datagen.gen_silesia_mix, "skewed": datagen.gen_skewed_bytes}[kind]
    plains = [bytes(gen(BLOCK, 1000 + s)) for s in range(16)]
    frames, res = batch(pkg, ctx, plains, pkg.LEVEL_FASTEST, checksum=False)
    ours = sum(len(f) for f in frames)
    ref = sum(len(datagen.compress(p, level=1, checksum=False)) for p in plains)
    print(f"{kind}: ours {ours} libzstd-1 {ref} ratio {ours / ref:.3f}")
    assert ours / ref <= gate


@pytest.mark.gpu
def test_short_out_cap_fails_only_that_frame(pkg, ctx):
    import datagen
    plains = [bytes(datagen.gen_text(100000, 40 + i)) for i in range(3)]
    caps = [pkg.compress_bound(len(p)) for p in plains]
    caps[1] = 100
    frames, res = batch(pkg, ctx, plains, pkg.LEVEL_FASTEST, out_caps=caps)
    assert res[1]["status"] == 18 and res[1]["out_size"] == 0   # TARGET_TOO_SMALL
    assert res[0]["status"] == 0 and res[2]["status"] == 0
    assert datagen.decompress(frames[0], len(plains[0])) == plains[0] and datagen.decompress(frames[2], len(plains[2])) == plains[2]


@pytest.mark.gpu
def test_levels_2_to_4_are_rejected(pkg, ctx):
    for level in (2, 3, 4):
        with pytest.raises(pkg.B200ZError) as e:
            pkg.compress(ctx, b"hello", level=level)
        assert e.value.code == 200
        io = np.array([(0, 5, 0, 64)], dtype=pkg.binding.FRAME_IO_DTYPE)
        assert ctx.L.b200z_compress_frames_batch(ctx.h, b"hello", 5, 0, io.ctypes.data, 1, level, 0, np.zeros(64, np.uint8).ctypes.data, 64, 0,
                                                 np.zeros(1, pkg.COMPRESS_RESULT_DTYPE).ctypes.data) == 200


@pytest.mark.gpu
def test_compress_through_read_and_write_callbacks(pkg, ctx, oracle):
    import io as _io
    import datagen
    p = bytes(datagen.gen_silesia_mix(1 << 20, 50))
    sink = _io.BytesIO()
    pkg.compress_stream(ctx, _io.BytesIO(p), sink)
    f = sink.getvalue()
    assert f == pkg.compress(ctx, p)
    assert oracle.decode_frame(f)[0] == p


@pytest.mark.gpu
@pytest.mark.slow
def test_c2b_gib_device_to_device(pkg, ctx):
    import torch
    import datagen
    fs = datagen.config_c2b()
    plain = torch.from_numpy(np.ascontiguousarray(fs.plain)).cuda()
    n = fs.nframes
    io = np.zeros(n, dtype=pkg.binding.FRAME_IO_DTYPE)
    bound = pkg.compress_bound(int(fs.out_size.max()))
    io["src_off"], io["src_size"] = fs.out_off, fs.out_size
    io["out_off"], io["out_cap"] = np.arange(n, dtype=np.uint64) * bound, bound
    out = torch.zeros(n * bound, dtype=torch.uint8, device="cuda")
    res = pkg.compress_frames(ctx, plain, io, out)
    assert (res["status"] == 0).all()
    dio = np.zeros(n, dtype=pkg.binding.FRAME_IO_DTYPE)
    dio["src_off"], dio["src_size"], dio["out_off"], dio["out_cap"] = io["out_off"], res["out_size"], fs.out_off, fs.out_size
    dec = torch.zeros(len(fs.plain), dtype=torch.uint8, device="cuda")
    dres = pkg.decode_frames(ctx, out, dio, dec)
    assert (dres["status"] == 0).all() and torch.equal(dec, plain)


@pytest.mark.gpu
def test_host_output_outside_written_frames_is_left_alone(pkg, ctx):
    """Only out_size bytes at each successful frame's out_off are written: gaps between frames and the room of a frame that
    failed with TARGET_TOO_SMALL keep what the caller had there, also after an earlier call left other bytes in device scratch."""
    import datagen
    plains = [bytes(datagen.gen_text(90000, 60 + i)) for i in range(3)]
    pkg.compress_frames(ctx, b"".join(plains), np.array([(0, 270000, 0, 400000)], dtype=pkg.binding.FRAME_IO_DTYPE),
                        np.zeros(400000, np.uint8))   # leaves other bytes in the context's device copy of the output
    bound = pkg.compress_bound(90000)
    io = np.zeros(3, dtype=pkg.binding.FRAME_IO_DTYPE)
    for i in range(3):
        io[i] = (90000 * i, 90000, 1000 + i * (bound + 5000), bound if i != 1 else 50)
    out = np.full(3 * (bound + 5000) + 1000, 0xAB, dtype=np.uint8)
    res = pkg.compress_frames(ctx, b"".join(plains), io, out)
    assert [int(r["status"]) for r in res] == [0, 18, 0]
    written = np.zeros(len(out), dtype=bool)
    for i in (0, 2):
        o = int(io[i]["out_off"])
        written[o:o + int(res[i]["out_size"])] = True
        assert datagen.decompress(out[o:o + int(res[i]["out_size"])].tobytes(), 90000) == plains[i]
    assert (out[~written] == 0xAB).all()


@pytest.mark.gpu
def test_compresses_on_every_visible_device(pkg):
    """Kernel attributes are set per device: a context on each GPU of the process compresses (Fastest needs 160 KB of dynamic
    shared memory per CTA)."""
    import torch
    import datagen
    p = bytes(datagen.gen_text(300000, 70))
    for dev in range(torch.cuda.device_count()):
        c = pkg.Context(dev)
        try:
            f = pkg.compress(c, p)
            assert datagen.decompress(f, len(p)) == p, dev
        finally:
            c.close()
