"""ctypes binding of libb200zstd.so + Python mirrors of ruzstd's FrameDecoder / StreamingDecoder.

Reference interface mirrored (all paths relative to ruzstd/src/decoding/):
  FrameDecoder            frame_decoder.rs:80-84, 154-627
  BlockDecodingStrategy   frame_decoder.rs:96-100
  StreamingDecoder        streaming_decoder.rs:45-156
Everything here is plumbing over the C ABI; no decoding happens in Python.
"""
import ctypes as C
import io
import os
import re
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200Z_LIB: development knob to load an experimental build of the same library (profiles/variants.sh); never a fallback
_SO = os.environ.get("B200Z_LIB") or os.path.join(_HERE, "libb200zstd.so")
_HEADER = os.path.join(_HERE, "..", "include", "b200zstd.h")

READ_FN = C.CFUNCTYPE(C.c_long, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t)
WRITE_FN = C.CFUNCTYPE(C.c_long, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t)

ALL, UPTO_BLOCKS, UPTO_BYTES = 0, 1, 2
MEM_HOST, MEM_DEVICE = 0, 1
ERR_SKIP_FRAME = 8
FLAG_CHECKSUM = 1
ERR_REFERENCE_WOULD_PANIC = 200
# CompressionLevel (encoding/mod.rs:47-68); Default / Better / Best are unimplemented!() in the reference
LEVEL_UNCOMPRESSED, LEVEL_FASTEST, LEVEL_DEFAULT, LEVEL_BETTER, LEVEL_BEST = 0, 1, 2, 3, 4
COMPRESS_CHECKSUM, COMPRESS_CONTENT_SIZE = 1, 2


class FrameIO(C.Structure):
    _fields_ = [("src_off", C.c_uint64), ("src_size", C.c_uint64), ("out_off", C.c_uint64), ("out_cap", C.c_uint64)]


class FrameResult(C.Structure):
    _fields_ = [("out_size", C.c_uint64), ("bytes_read", C.c_uint64), ("content_size", C.c_uint64), ("window_size", C.c_uint64),
                ("status", C.c_int32), ("stage", C.c_int32), ("blocks_decoded", C.c_uint32), ("error_block", C.c_uint32),
                ("has_checksum", C.c_uint32), ("checksum_from_data", C.c_uint32), ("has_dict_id", C.c_uint32), ("dict_id", C.c_uint32),
                ("has_calculated_checksum", C.c_uint32), ("calculated_checksum", C.c_uint32)]


FRAME_IO_DTYPE = np.dtype([("src_off", "<u8"), ("src_size", "<u8"), ("out_off", "<u8"), ("out_cap", "<u8")])
BLOCK_DESC_DTYPE = np.dtype([("src_off", "<u8"), ("content_size", "<u4"), ("block_type", "<u4"), ("decompressed_size", "<u4"), ("last_block", "<u4"),
                             ("literals_type", "<u4"), ("regenerated_size", "<u4"), ("compressed_size", "<u4"), ("num_streams", "<u4"),
                             ("num_sequences", "<u4"), ("modes", "<u4")])
BLOCK_FRAME_DTYPE = np.dtype([("out_off", "<u8"), ("out_cap", "<u8"), ("window_size", "<u8"), ("dict", "<u8"), ("first_block", "<u4"), ("num_blocks", "<u4")])
BLOCK_STATUS_DTYPE = np.dtype([("status", "<i4"), ("stage", "<i4"), ("out_size", "<u4"), ("reserved", "<u4")])
BLOCK_NOT_REACHED = -1
FRAME_RESULT_DTYPE = np.dtype([("out_size", "<u8"), ("bytes_read", "<u8"), ("content_size", "<u8"), ("window_size", "<u8"),
                               ("status", "<i4"), ("stage", "<i4"), ("blocks_decoded", "<u4"), ("error_block", "<u4"),
                               ("has_checksum", "<u4"), ("checksum_from_data", "<u4"), ("has_dict_id", "<u4"), ("dict_id", "<u4"),
                               ("has_calculated_checksum", "<u4"), ("calculated_checksum", "<u4")])
COMPRESS_RESULT_DTYPE = np.dtype([("out_size", "<u8"), ("status", "<i4"), ("stage", "<i4"), ("num_blocks", "<u4"), ("raw_blocks", "<u4"),
                                  ("rle_blocks", "<u4"), ("compressed_blocks", "<u4"), ("checksum", "<u4"), ("reserved", "<u4")])
assert FRAME_IO_DTYPE.itemsize == C.sizeof(FrameIO) and FRAME_RESULT_DTYPE.itemsize == C.sizeof(FrameResult)


def lib_path():
    return _SO


def build(force=False):
    """Compile libb200zstd.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))] + [_HEADER, os.path.join(_HERE, "Makefile")]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs):
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return _SO


_lib = None


def lib():
    """The loaded library.  Raises if it was not built -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise RuntimeError(f"{_SO} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)")
    L = C.CDLL(_SO)
    vp, sz, u8p = C.c_void_p, C.c_size_t, C.POINTER(C.c_uint8)
    pp = C.POINTER(vp)
    sig = {
        "b200z_error_name": (C.c_char_p, [C.c_int]),
        "b200z_abi_version": (C.c_int, []),
        "b200z_ctx_create": (C.c_int, [C.c_int, pp]),
        "b200z_ctx_destroy": (None, [vp]),
        "b200z_ctx_last_error_message": (C.c_char_p, [vp]),
        "b200z_ctx_stream": (vp, [vp]),
        "b200z_ctx_kernel_launches": (C.c_uint64, [vp]),
        "b200z_ctx_set_flags": (None, [vp, C.c_uint32]),
        "b200z_ctx_flags": (C.c_uint32, [vp]),
        "b200z_dict_create": (C.c_int, [vp, vp, sz, pp]),
        "b200z_dict_create_raw_content": (C.c_int, [vp, C.c_uint32, vp, sz, pp]),
        "b200z_dict_id": (C.c_uint32, [vp]),
        "b200z_dict_offset_history": (C.c_int, [vp, C.POINTER(C.c_uint32)]),
        "b200z_dict_content_size": (sz, [vp]),
        "b200z_dict_destroy": (None, [vp]),
        "b200z_decode_frames_batch": (C.c_int, [vp, vp, sz, C.c_int, vp, sz, pp, sz, vp, C.c_uint64, vp, sz, C.c_int, vp]),
        "b200z_decode_blocks_batch": (C.c_int, [vp, vp, sz, vp, sz, vp, sz, C.c_int, vp, sz, C.c_int, vp, vp]),
        "b200z_batch_prepare": (C.c_int, [vp, vp, sz, C.c_int, vp, sz, pp, sz, vp, C.c_uint64, pp]),
        "b200z_batch_run": (C.c_int, [vp, vp, sz]),
        "b200z_batch_finish": (C.c_int, [vp, vp]),
        "b200z_batch_run_profile": (C.c_int, [vp, vp, sz, C.POINTER(C.c_float), sz]),
        "b200z_batch_run_timeline": (C.c_int, [vp, vp, sz, C.POINTER(C.c_float), sz]),
        "b200z_num_stages": (C.c_int, []),
        "b200z_stage_kernel_name": (C.c_char_p, [C.c_int]),
        "b200z_batch_info": (C.c_int, [vp, C.POINTER(C.c_uint64)]),
        "b200z_batch_debug_literals": (C.c_int, [vp, C.c_uint32, vp, sz, C.POINTER(sz)]),
        "b200z_batch_debug_sequences": (C.c_int, [vp, C.c_uint32, vp, sz, C.POINTER(sz)]),
        "b200z_batch_debug_block_flags": (C.c_int, [vp, C.c_uint32, C.POINTER(C.c_uint32)]),
        "b200z_batch_debug_sched": (C.c_int, [vp, C.POINTER(C.c_uint32)]),
        "b200z_debug_route_frames": (C.c_int, [vp, vp, sz, C.c_uint32, vp, C.POINTER(sz)]),
        "b200z_debug_fse_order": (C.c_int, [vp, vp, vp, sz, vp, sz, vp, C.POINTER(sz)]),
        "b200z_batch_destroy": (None, [vp]),
        "b200z_frame_decoder_new": (C.c_int, [vp, pp]),
        "b200z_frame_decoder_free": (None, [vp]),
        "b200z_frame_decoder_set_max_window_size": (None, [vp, C.c_uint64]),
        "b200z_frame_decoder_max_window_size": (C.c_uint64, [vp]),
        "b200z_frame_decoder_init": (C.c_int, [vp, READ_FN, vp]),
        "b200z_frame_decoder_reset": (C.c_int, [vp, READ_FN, vp]),
        "b200z_frame_decoder_skip_frame_length": (C.c_uint32, [vp]),
        "b200z_frame_decoder_add_dict": (C.c_int, [vp, vp, sz]),
        "b200z_frame_decoder_add_raw_content_dict": (C.c_int, [vp, C.c_uint32, vp, sz]),
        "b200z_frame_decoder_force_dict": (C.c_int, [vp, C.c_uint32]),
        "b200z_frame_decoder_decode_blocks": (C.c_int, [vp, READ_FN, vp, C.c_int, sz, C.POINTER(C.c_int)]),
        "b200z_frame_decoder_read": (C.c_long, [vp, vp, sz]),
        "b200z_frame_decoder_collect_to_writer": (C.c_long, [vp, WRITE_FN, vp]),
        "b200z_frame_decoder_can_collect": (sz, [vp]),
        "b200z_frame_decoder_is_finished": (C.c_int, [vp]),
        "b200z_frame_decoder_blocks_decoded": (sz, [vp]),
        "b200z_frame_decoder_bytes_read_from_source": (C.c_uint64, [vp]),
        "b200z_frame_decoder_content_size": (C.c_uint64, [vp]),
        "b200z_frame_decoder_get_checksum_from_data": (C.c_int, [vp, C.POINTER(C.c_uint32)]),
        "b200z_frame_decoder_get_calculated_checksum": (C.c_int, [vp, C.POINTER(C.c_uint32)]),
        "b200z_frame_decoder_decode_from_to": (C.c_int, [vp, vp, sz, vp, sz, C.POINTER(sz), C.POINTER(sz)]),
        "b200z_frame_decoder_decode_all": (C.c_int, [vp, vp, sz, vp, sz, C.POINTER(sz)]),
        "b200z_frame_decoder_last_stage": (C.c_int, [vp]),
        "b200z_frame_decoder_last_error_message": (C.c_char_p, [vp]),
        "b200z_streaming_decoder_new": (C.c_int, [vp, READ_FN, vp, pp]),
        "b200z_streaming_decoder_new_with_decoder": (C.c_int, [READ_FN, vp, vp, pp]),
        "b200z_streaming_decoder_new_with_max_window_size": (C.c_int, [vp, READ_FN, vp, C.c_uint64, pp]),
        "b200z_streaming_decoder_read": (C.c_long, [vp, vp, sz, C.POINTER(C.c_int)]),
        "b200z_streaming_decoder_frame_decoder": (vp, [vp]),
        "b200z_streaming_decoder_into_frame_decoder": (vp, [vp]),
        "b200z_streaming_decoder_free": (None, [vp]),
        "b200z_xxh64": (C.c_uint64, [vp, sz]),
        "b200z_compress_bound": (sz, [sz]),
        "b200z_compress_frames_batch": (C.c_int, [vp, vp, sz, C.c_int, vp, sz, C.c_int, C.c_uint32, vp, sz, C.c_int, vp]),
        "b200z_compress": (C.c_int, [vp, READ_FN, vp, WRITE_FN, vp, C.c_int, C.c_uint32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)          # AttributeError here == a symbol the header declares is not exported
        fn.restype = res
        fn.argtypes = args
    L._declared = sorted(sig)
    _lib = L
    return L


def declared_symbols():
    """Every function include/b200zstd.h declares (parsed from the header)."""
    txt = open(_HEADER).read()
    return sorted(set(re.findall(r"\b(b200z_[a-z0-9_]+)\s*\(", txt)))


def error_names():
    txt = open(_HEADER).read()
    return {int(v): k for k, v in re.findall(r"(B200Z_(?:OK|ERR_[A-Z0-9_]+))\s*=\s*(\d+)", txt)}


class B200ZError(Exception):
    """Mirror of ruzstd's FrameDecoderError: .code is the leaf variant, .stage the nesting path."""

    def __init__(self, code, stage=0, msg=""):
        self.code, self.stage = code, stage
        super().__init__(f"{lib().b200z_error_name(code).decode()} (stage {stage}) {msg}")


def xxh64(data):
    b = bytes(data)
    return lib().b200z_xxh64(b, len(b))


def route_frames(work, eligible, sms=148):
    """Host-only: the frames k_exec_cta would take (largest first) -- route_exec_frames, csrc/plan.cpp."""
    w = np.ascontiguousarray(work, dtype=np.uint64)
    el = np.ascontiguousarray(eligible, dtype=np.uint8)
    out = np.zeros(max(len(w), 1), dtype=np.uint32)
    n = C.c_size_t()
    rc = lib().b200z_debug_route_frames(w.ctypes.data, el.ctypes.data, len(w), sms, out.ctypes.data, C.byref(n))
    if rc:
        raise B200ZError(rc, 0, "b200z_debug_route_frames")
    return out[:n.value].copy()


def fse_order(first_block, nblocks, on_cta, nseq):
    """Host-only: the order in which k_fse takes the blocks (empty = descriptor order) -- build_fse_order, csrc/plan.cpp."""
    fb = np.ascontiguousarray(first_block, dtype=np.uint32)
    nb = np.ascontiguousarray(nblocks, dtype=np.uint32)
    oc = np.ascontiguousarray(on_cta, dtype=np.uint8)
    ns = np.ascontiguousarray(nseq, dtype=np.uint32)
    out = np.zeros(max(len(ns), 1), dtype=np.uint32)
    n = C.c_size_t()
    rc = lib().b200z_debug_fse_order(fb.ctypes.data, nb.ctypes.data, oc.ctypes.data, len(fb), ns.ctypes.data, len(ns), out.ctypes.data, C.byref(n))
    if rc:
        raise B200ZError(rc, 0, "b200z_debug_fse_order")
    return out[:n.value].copy()


def _ptr(x):
    """(address, nbytes, keepalive) of bytes / numpy / torch tensor (host or device)."""
    if x is None:
        return None, 0, None
    if isinstance(x, (bytes, bytearray)):
        a = np.frombuffer(x, dtype=np.uint8)
        return a.ctypes.data, a.nbytes, a
    if isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x)
        return a.ctypes.data, a.nbytes, a
    if hasattr(x, "data_ptr"):  # torch tensor
        return x.data_ptr(), x.numel() * x.element_size(), x
    raise TypeError(type(x))


def _is_device(x):
    return hasattr(x, "is_cuda") and x.is_cuda


class Context:
    """One per GPU: pins the device, owns the stream (b200z_ctx)."""

    def __init__(self, device=0):
        self.L = lib()
        h = C.c_void_p()
        e = self.L.b200z_ctx_create(device, C.byref(h))
        if e:
            raise B200ZError(e, 0, "b200z_ctx_create: no usable CUDA device; this library has no CPU path")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.b200z_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def stream(self):
        return self.L.b200z_ctx_stream(self.h)

    def kernel_launches(self):
        return self.L.b200z_ctx_kernel_launches(self.h)

    def set_flags(self, flags):
        """FLAG_CHECKSUM = 1: the batch entry also computes each frame's XXH64 content checksum on the GPU."""
        self.L.b200z_ctx_set_flags(self.h, flags)

    def _chk(self, e):
        if e:
            raise B200ZError(e, 0, self.L.b200z_ctx_last_error_message(self.h).decode())


class Dictionary:
    """Mirror of ruzstd::decoding::Dictionary (dictionary.rs:12-37); decode_dict == Dictionary.decode_dict."""

    def __init__(self, ctx, handle):
        self.ctx, self.h = ctx, handle

    @classmethod
    def decode_dict(cls, ctx, raw):
        h = C.c_void_p()
        b = bytes(raw)
        e = ctx.L.b200z_dict_create(ctx.h, b, len(b), C.byref(h))
        if e:
            raise B200ZError(e, 8)
        return cls(ctx, h)

    @classmethod
    def raw_content(cls, ctx, dict_id, content):
        h = C.c_void_p()
        b = bytes(content)
        ctx._chk(ctx.L.b200z_dict_create_raw_content(ctx.h, dict_id, b, len(b), C.byref(h)))
        return cls(ctx, h)

    @property
    def id(self):
        return self.ctx.L.b200z_dict_id(self.h)

    @property
    def offset_hist(self):
        a = (C.c_uint32 * 3)()
        self.ctx.L.b200z_dict_offset_history(self.h, a)
        return list(a)

    @property
    def content_size(self):
        return self.ctx.L.b200z_dict_content_size(self.h)

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                self.ctx.L.b200z_dict_destroy(self.h)
        except Exception:
            pass


def _frames_array(frames):
    a = np.ascontiguousarray(frames, dtype=FRAME_IO_DTYPE) if not (isinstance(frames, np.ndarray) and frames.dtype == FRAME_IO_DTYPE) else np.ascontiguousarray(frames)
    return a


def _dict_args(dicts, forced):
    dicts = list(dicts or [])
    arr = (C.c_void_p * max(len(dicts), 1))(*[d.h for d in dicts])
    return arr, len(dicts), (forced.h if forced is not None else None)


def decode_blocks(ctx, blocks, frames, compressed, output):
    """b200z_decode_blocks_batch: the block-level entry (what replaces BlockDecoder::decompress_block, block_decoder.rs:97-197).
    blocks: BLOCK_DESC_DTYPE array, frames: BLOCK_FRAME_DTYPE array ('dict' = Dictionary or 0 per frame via `set_frame_dicts`).
    Returns (block status array, per-frame output sizes)."""
    blocks = np.ascontiguousarray(blocks, dtype=BLOCK_DESC_DTYPE)
    frames = np.ascontiguousarray(frames, dtype=BLOCK_FRAME_DTYPE)
    st = np.zeros(len(blocks), dtype=BLOCK_STATUS_DTYPE)
    fo = np.zeros(len(frames), dtype=np.uint64)
    ip, il, _k1 = _ptr(compressed)
    op, ol, _k2 = _ptr(output)
    e = ctx.L.b200z_decode_blocks_batch(ctx.h, blocks.ctypes.data, len(blocks), frames.ctypes.data, len(frames), ip, il,
                                        MEM_DEVICE if _is_device(compressed) else MEM_HOST, op, ol, MEM_DEVICE if _is_device(output) else MEM_HOST,
                                        st.ctypes.data, fo.ctypes.data)
    ctx._chk(e)
    return st, fo


def decode_frames(ctx, input, frames, output, dicts=None, forced_dict=None, max_window_size=0):
    """b200z_decode_frames_batch: one-shot batch decode.  input/output: bytes, numpy or torch (host or cuda)."""
    fr = _frames_array(frames)
    res = np.zeros(len(fr), dtype=FRAME_RESULT_DTYPE)
    ip, il, _k1 = _ptr(input)
    op, ol, _k2 = _ptr(output)
    darr, nd, forced = _dict_args(dicts, forced_dict)
    e = ctx.L.b200z_decode_frames_batch(ctx.h, ip, il, MEM_DEVICE if _is_device(input) else MEM_HOST, fr.ctypes.data, len(fr),
                                        darr, nd, forced, max_window_size, op, ol, MEM_DEVICE if _is_device(output) else MEM_HOST,
                                        res.ctypes.data)
    ctx._chk(e)
    return res


def compress_bound(n):
    """b200z_compress_bound: the largest frame compress_frames writes for n plaintext bytes."""
    return lib().b200z_compress_bound(n)


def _check_level(level):
    if level in (LEVEL_DEFAULT, LEVEL_BETTER, LEVEL_BEST):   # frame_compressor.rs:202-204: unimplemented!()
        raise B200ZError(ERR_REFERENCE_WOULD_PANIC, 0, f"compression level {level} is not implemented by the reference")
    if level not in (LEVEL_UNCOMPRESSED, LEVEL_FASTEST):
        raise ValueError(f"unknown compression level {level}")


def _compress_flags(checksum, content_size):
    return (COMPRESS_CHECKSUM if checksum else 0) | (COMPRESS_CONTENT_SIZE if content_size else 0)


def compress_frames(ctx, input, frames, output, level=LEVEL_FASTEST, checksum=True, content_size=False):
    """b200z_compress_frames_batch: many independent frames at once.  frames: FRAME_IO_DTYPE rows {src_off, src_size, out_off,
    out_cap} (src = plaintext inside `input`, out = where the frame goes inside `output`); input/output: bytes, numpy or torch
    (host or cuda).  Returns a COMPRESS_RESULT_DTYPE array."""
    _check_level(level)
    fr = _frames_array(frames)
    res = np.zeros(len(fr), dtype=COMPRESS_RESULT_DTYPE)
    ip, il, _k1 = _ptr(input)
    op, ol, _k2 = _ptr(output)
    e = ctx.L.b200z_compress_frames_batch(ctx.h, ip, il, MEM_DEVICE if _is_device(input) else MEM_HOST, fr.ctypes.data, len(fr), level,
                                          _compress_flags(checksum, content_size), op, ol, MEM_DEVICE if _is_device(output) else MEM_HOST,
                                          res.ctypes.data)
    ctx._chk(e)
    return res


def compress(ctx, data, level=LEVEL_FASTEST, checksum=True, content_size=False):
    """encoding::compress_to_vec (mod.rs:33-37): one frame for `data`, as bytes."""
    _check_level(level)
    src = bytes(data)
    cap = compress_bound(len(src))
    out = np.empty(cap, dtype=np.uint8)
    io = np.array([(0, len(src), 0, cap)], dtype=FRAME_IO_DTYPE)
    r = compress_frames(ctx, src, io, out, level, checksum, content_size)[0]
    if r["status"]:
        raise B200ZError(int(r["status"]), int(r["stage"]))
    return out[:int(r["out_size"])].tobytes()


def compress_stream(ctx, reader, writer, level=LEVEL_FASTEST, checksum=True, content_size=False):
    """b200z_compress == encoding::compress(source, target, level) (mod.rs:24-30): reader.read(n) to EOF, writer.write(b)."""
    _check_level(level)

    def _rd(_user, buf, n):
        b = reader.read(n)
        if b:
            C.memmove(buf, b, len(b))
        return len(b)

    def _wr(_user, buf, n):
        return writer.write(C.string_at(buf, n)) or 0
    rcb, wcb = READ_FN(_rd), WRITE_FN(_wr)
    ctx._chk(ctx.L.b200z_compress(ctx.h, rcb, None, wcb, None, level, _compress_flags(checksum, content_size)))


class Batch:
    """Prepared submission: plan + descriptors + input resident in HBM; run() launches kernels only."""

    def __init__(self, ctx, input, frames, dicts=None, forced_dict=None, max_window_size=0):
        self.ctx = ctx
        self.frames = _frames_array(frames)
        ip, il, self._k = _ptr(input)
        darr, nd, forced = _dict_args(dicts, forced_dict)
        self._dicts = (dicts, forced_dict)
        h = C.c_void_p()
        ctx._chk(ctx.L.b200z_batch_prepare(ctx.h, ip, il, MEM_DEVICE if _is_device(input) else MEM_HOST, self.frames.ctypes.data,
                                           len(self.frames), darr, nd, forced, max_window_size, C.byref(h)))
        self.h = h

    def run(self, d_output):
        op, ol, _k = _ptr(d_output)
        assert _is_device(d_output), "Batch.run writes into device memory"
        self.ctx._chk(self.ctx.L.b200z_batch_run(self.h, op, ol))

    def run_profile(self, d_output):
        """{kernel name: device ms} for one pass, measured with CUDA events between the kernels."""
        op, ol, _k = _ptr(d_output)
        n = self.ctx.L.b200z_num_stages()
        ms = (C.c_float * n)()
        self.ctx._chk(self.ctx.L.b200z_batch_run_profile(self.h, op, ol, ms, n))
        return {self.ctx.L.b200z_stage_kernel_name(i).decode(): float(ms[i]) for i in range(n)}

    def run_timeline(self, d_output):
        """Completion time (ms from the start of the pass) of each kernel in the overlapped launch."""
        op, ol, _k = _ptr(d_output)
        ms = (C.c_float * 4)()
        self.ctx._chk(self.ctx.L.b200z_batch_run_timeline(self.h, op, ol, ms, 4))
        return {"k_setup+k_huf": float(ms[1]), "k_fse+k_exec": float(ms[2]), "k_exec_cta+k_exec": float(ms[3])}

    def finish(self):
        res = np.zeros(len(self.frames), dtype=FRAME_RESULT_DTYPE)
        self.ctx._chk(self.ctx.L.b200z_batch_finish(self.h, res.ctypes.data))
        return res

    def info(self):
        a = (C.c_uint64 * 8)()
        self.ctx.L.b200z_batch_info(self.h, a)
        k = ["frames", "blocks", "compressed_blocks", "planned_bytes", "literal_scratch_bytes", "sequences", "launches_per_run"]
        return dict(zip(k, list(a)))

    def debug_literals(self, block, cap=1 << 20):
        buf = np.empty(cap, dtype=np.uint8)
        n = C.c_size_t()
        self.ctx._chk(self.ctx.L.b200z_batch_debug_literals(self.h, block, buf.ctypes.data, cap, C.byref(n)))
        return buf[:n.value].tobytes()

    def debug_sequences(self, block, cap=100000):
        buf = np.empty((cap, 3), dtype=np.uint32)
        n = C.c_size_t()
        self.ctx._chk(self.ctx.L.b200z_batch_debug_sequences(self.h, block, buf.ctypes.data, cap, C.byref(n)))
        return buf[:n.value].copy()

    def debug_sched(self):
        a = (C.c_uint32 * 4)()
        self.ctx._chk(self.ctx.L.b200z_batch_debug_sched(self.h, a))
        return {"cta_frames": a[0], "handed_back_frames": a[1], "reasons": a[2], "handed_back_blocks": a[3]}

    def debug_block_flags(self, block):
        v = C.c_uint32()
        self.ctx._chk(self.ctx.L.b200z_batch_debug_block_flags(self.h, block, C.byref(v)))
        return v.value

    def close(self):
        if getattr(self, "h", None) and self.ctx.h:
            self.ctx.L.b200z_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Reader:
    """io::Read adaptor over bytes or a Python file-like; keeps the ctypes callback alive."""

    def __init__(self, src):
        if isinstance(src, (bytes, bytearray, memoryview)):
            src = io.BytesIO(bytes(src))
        self.src = src

        def _cb(_user, buf, n):
            b = self.src.read(n)
            if b:
                C.memmove(buf, b, len(b))
            return len(b)
        self.cb = READ_FN(_cb)


class FrameDecoder:
    """GPU-backed mirror of ruzstd::decoding::FrameDecoder (frame_decoder.rs:154-627)."""

    def __init__(self, ctx, _handle=None):
        self.ctx, self.L = ctx, ctx.L
        if _handle is None:
            h = C.c_void_p()
            ctx._chk(self.L.b200z_frame_decoder_new(ctx.h, C.byref(h)))
            _handle = h
        self.h = _handle

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                self.L.b200z_frame_decoder_free(self.h)
        except Exception:
            pass

    def _chk(self, e):
        if e:
            raise B200ZError(e, self.L.b200z_frame_decoder_last_stage(self.h), self.L.b200z_frame_decoder_last_error_message(self.h).decode())

    def set_max_window_size(self, n): self.L.b200z_frame_decoder_set_max_window_size(self.h, n)
    def max_window_size(self): return self.L.b200z_frame_decoder_max_window_size(self.h)

    def reset(self, reader):
        if not isinstance(reader, _Reader):
            reader = _Reader(reader)
        self._chk(self.L.b200z_frame_decoder_reset(self.h, reader.cb, None))
        return reader
    init = reset

    def skip_frame_length(self): return self.L.b200z_frame_decoder_skip_frame_length(self.h)

    def add_dict(self, raw):
        b = bytes(raw)
        self._chk(self.L.b200z_frame_decoder_add_dict(self.h, b, len(b)))

    def add_raw_content_dict(self, dict_id, content):
        b = bytes(content)
        self._chk(self.L.b200z_frame_decoder_add_raw_content_dict(self.h, dict_id, b, len(b)))

    def force_dict(self, dict_id): self._chk(self.L.b200z_frame_decoder_force_dict(self.h, dict_id))

    def decode_blocks(self, reader, strategy=ALL, n=0):
        fin = C.c_int(0)
        self._chk(self.L.b200z_frame_decoder_decode_blocks(self.h, reader.cb, None, strategy, n, C.byref(fin)))
        return bool(fin.value)

    def read(self, n):
        buf = np.empty(max(n, 1), dtype=np.uint8)
        r = self.L.b200z_frame_decoder_read(self.h, buf.ctypes.data, n)
        if r < 0:
            raise B200ZError(16, 9)
        return buf[:r].tobytes()

    def collect(self):
        """FrameDecoder::collect (frame_decoder.rs:381-389)."""
        out = bytearray()
        while True:
            n = self.can_collect()
            if n == 0:
                return bytes(out)
            out += self.read(n)

    def collect_to_writer(self, writer):
        def _cb(_user, buf, n):
            return writer.write(C.string_at(buf, n)) or 0
        cb = WRITE_FN(_cb)
        r = self.L.b200z_frame_decoder_collect_to_writer(self.h, cb, None)
        if r < 0:
            raise B200ZError(16, 9)
        return r

    def can_collect(self): return self.L.b200z_frame_decoder_can_collect(self.h)
    def is_finished(self): return bool(self.L.b200z_frame_decoder_is_finished(self.h))
    def blocks_decoded(self): return self.L.b200z_frame_decoder_blocks_decoded(self.h)
    def bytes_read_from_source(self): return self.L.b200z_frame_decoder_bytes_read_from_source(self.h)
    def content_size(self): return self.L.b200z_frame_decoder_content_size(self.h)

    def get_checksum_from_data(self):
        v = C.c_uint32()
        return v.value if self.L.b200z_frame_decoder_get_checksum_from_data(self.h, C.byref(v)) else None

    def get_calculated_checksum(self):
        v = C.c_uint32()
        return v.value if self.L.b200z_frame_decoder_get_calculated_checksum(self.h, C.byref(v)) else None

    def decode_from_to(self, source, target_len):
        src = bytes(source)
        buf = np.empty(max(target_len, 1), dtype=np.uint8)
        r, w = C.c_size_t(), C.c_size_t()
        self._chk(self.L.b200z_frame_decoder_decode_from_to(self.h, src, len(src), buf.ctypes.data, target_len, C.byref(r), C.byref(w)))
        return r.value, buf[:w.value].tobytes()

    def decode_all(self, data, out_cap):
        src = bytes(data)
        buf = np.empty(max(out_cap, 1), dtype=np.uint8)
        w = C.c_size_t()
        self._chk(self.L.b200z_frame_decoder_decode_all(self.h, src, len(src), buf.ctypes.data, out_cap, C.byref(w)))
        return buf[:w.value].tobytes()

    def decode_all_to_vec(self, data, capacity):
        """decode_all_to_vec (frame_decoder.rs:591-610): `capacity` plays the Vec's spare capacity."""
        return self.decode_all(data, capacity)


class StreamingDecoder:
    """GPU-backed mirror of ruzstd::decoding::StreamingDecoder (streaming_decoder.rs:45-156)."""

    def __init__(self, ctx, source, decoder=None, max_window_size=None):
        self.ctx, self.L = ctx, ctx.L
        self.source = _Reader(source)
        h = C.c_void_p()
        self._borrowed = decoder
        if decoder is not None:        # new_with_decoder
            e = self.L.b200z_streaming_decoder_new_with_decoder(self.source.cb, None, decoder.h, C.byref(h))
            if e:
                raise B200ZError(e, self.L.b200z_frame_decoder_last_stage(decoder.h))
        elif max_window_size is not None:
            e = self.L.b200z_streaming_decoder_new_with_max_window_size(ctx.h, self.source.cb, None, max_window_size, C.byref(h))
            if e:
                raise B200ZError(e, 1)
        else:
            e = self.L.b200z_streaming_decoder_new(ctx.h, self.source.cb, None, C.byref(h))
            if e:
                raise B200ZError(e, 1)
        self.h = h

    def read(self, n):
        buf = np.empty(max(n, 1), dtype=np.uint8)
        err = C.c_int(0)
        r = self.L.b200z_streaming_decoder_read(self.h, buf.ctypes.data, n, C.byref(err))
        if r < 0:
            raise B200ZError(err.value or 16)
        return buf[:r].tobytes()

    def read_to_end(self, chunk=1 << 16):
        out = bytearray()
        while True:
            b = self.read(chunk)
            if not b:
                return bytes(out)
            out += b

    def into_frame_decoder(self):
        if self._borrowed is not None:
            self.L.b200z_streaming_decoder_free(self.h); self.h = None
            return self._borrowed
        dh = self.L.b200z_streaming_decoder_into_frame_decoder(self.h)
        self.h = None
        return FrameDecoder(self.ctx, C.c_void_p(dh))

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                self.L.b200z_streaming_decoder_free(self.h)
        except Exception:
            pass
