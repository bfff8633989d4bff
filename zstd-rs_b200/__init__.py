"""zstd-rs_b200 -- B200-native zstd decompressor and compressor behind ruzstd's FrameDecoder / StreamingDecoder / compress API.

The product is the C-ABI library ``libb200zstd.so`` (include/b200zstd.h, sources in csrc/).  This package is the
Python host-side mirror of the reference interface (same names, argument meaning and error behaviour as
ruzstd::decoding::{FrameDecoder, StreamingDecoder, BlockDecodingStrategy}) over that ABI via ctypes.

There is no CPU decode or compression path: every call needs a CUDA device and fails loudly without one.
Import name: ``zstd_rs_b200`` (the directory name has a hyphen; see ``_pkg.py`` at the repo root).
"""
from .binding import (  # noqa: F401
    ALL, COMPRESS_RESULT_DTYPE, LEVEL_BEST, LEVEL_BETTER, LEVEL_DEFAULT, LEVEL_FASTEST, LEVEL_UNCOMPRESSED, UPTO_BLOCKS, UPTO_BYTES,
    B200ZError, Batch, Context, Dictionary, FrameDecoder, StreamingDecoder, build, compress, compress_bound, compress_frames,
    compress_stream, decode_blocks, decode_frames, error_names, lib, lib_path, xxh64,
)
from . import binding  # noqa: F401
