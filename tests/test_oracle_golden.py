"""Pins the CPU oracle (oracle/ruzstd_oracle.c) against every golden vector the reference's own tests hold for the
decode path (SURVEY.md 8c) and against libzstd as a secondary oracle.  CPU only."""
import hashlib

import numpy as np
import pytest

from conftest import golden_path, read_golden


def test_decode_corpus(oracle, manifest):
    """ruzstd/src/tests/decode_corpus.rs:1-189: size, byte equality, bytes_read == file size, checksum equality."""
    assert len(manifest["corpus"]) == 101
    for name, m in manifest["corpus"].items():
        data = read_golden("decodecorpus", name)
        out, d = oracle.decode_frame(data)
        assert len(out) == m["size"], name
        assert hashlib.sha256(out).hexdigest() == m["sha256"], name
        assert d.bytes_read_from_source() == len(data), name
        assert d.get_checksum_from_data() is not None and d.get_checksum_from_data() == d.get_calculated_checksum() == m["xxh64_low32"], name
        assert d.is_finished()


def test_decode_corpus_against_reference_originals(oracle, manifest):
    """Same as above but byte-for-byte against windows of the reference's original files (decodecorpus_originals.npz,
    written by make_golden.py: every original of up to 256 bytes whole, else its head, its tail and four seeded windows)."""
    z = np.load(golden_path("decodecorpus_originals.npz"), allow_pickle=False)
    assert sorted(z["name"]) == sorted(manifest["corpus"])
    out = {name: oracle.decode_frame(read_golden("decodecorpus", name))[0] for name in z["name"]}
    for name, size in zip(z["name"], z["size"]):
        assert len(out[name]) == size, name
    ends = np.cumsum(z["win_len"], dtype=np.uint64)
    for f, o, n, e in zip(z["win_file"], z["win_off"], z["win_len"], ends):
        name = z["name"][f]
        assert out[name][o:o + n] == z["val"][e - n:e].tobytes(), (name, int(o))


def test_dict_corpus(oracle, manifest):
    """ruzstd/src/tests/dict_test.rs:77-262."""
    dic = read_golden("dict_tests", "dictionary")
    assert len(manifest["dict"]) == 207
    for name, m in manifest["dict"].items():
        data = read_golden("dict_tests", "files", name)
        out, d = oracle.decode_frame(data, dict_raw=dic)
        assert len(out) == m["size"] and hashlib.sha256(out).hexdigest() == m["sha256"], name
        assert d.bytes_read_from_source() == len(data), name


def test_window_fixtures(oracle, manifest):
    """ruzstd/src/tests/mod.rs:576-741 window-limit tests."""
    fox = b"The quick brown fox jumps over the lazy dog.\n" * 4096
    big = read_golden("test_fixtures", "window_256mib.zst")
    small = read_golden("test_fixtures", "window_8mib.zst")
    d = oracle.FrameDecoder()
    d.set_max_window_size(300 << 20)
    assert d.max_window_size() == 300 << 20
    assert d.decode_all(big, len(fox)) == fox
    d = oracle.FrameDecoder()
    assert d.max_window_size() == 128 << 20
    with pytest.raises(oracle.OracleError) as e:
        d.decode_all(big, len(fox))
    assert oracle.error_names()[e.value.code] == "ZO_ERR_WINDOW_SIZE_TOO_BIG"
    d = oracle.FrameDecoder(); d.set_max_window_size(300 << 20)
    assert d.decode_all(big + big, 2 * len(fox)) == fox + fox
    d = oracle.FrameDecoder()
    with pytest.raises(oracle.OracleError):
        d.decode_all(small + big, 1 << 20)
    d = oracle.FrameDecoder()
    d.set_max_window_size(2 ** 64 - 1)
    assert d.max_window_size() == (1 << 41) + 7 * (1 << 38)
    for name, m in manifest["fixtures"].items():
        d = oracle.FrameDecoder(); d.set_max_window_size(300 << 20)
        out = d.decode_all(read_golden("test_fixtures", name), m["size"] + 8)
        assert hashlib.sha256(out).hexdigest() == m["sha256"], name


def test_fuzz_artifacts_do_not_crash(oracle, manifest):
    """ruzstd/src/tests/fuzz_regressions.rs: errors are fine, crashes are not."""
    n = 0
    for sub, files in manifest["fuzz"].items():
        for f in files:
            data = read_golden("fuzz", sub, f)
            try:
                oracle.decode_frame(data)
            except oracle.OracleError:
                pass
            n += 1
    assert n == 49


def test_api_decode_from_to(oracle, manifest):
    """tests/mod.rs:129-230: split input, checksum-only tail."""
    content = read_golden("decodecorpus", "z000088.zst")
    d = oracle.FrameDecoder()
    read1, out1 = d.decode_from_to(content[:50 * 1024], 1 << 20)
    read2, out2 = d.decode_from_to(content[read1:len(content) - 4], 1 << 20)
    assert read1 + read2 == len(content) - 4
    read3, out3 = d.decode_from_to(content[read1 + read2:], 1 << 20)
    assert read3 == 4 and out3 == b""
    res = out1 + out2
    m = manifest["corpus"]["z000088.zst"]
    assert len(res) == m["size"] and hashlib.sha256(res).hexdigest() == m["sha256"]
    assert d.get_checksum_from_data() == d.get_calculated_checksum()


def test_api_streaming_and_reuse(oracle, manifest):
    """tests/mod.rs:294-380: StreamingDecoder + new_with_decoder reuse."""
    s = oracle.StreamingDecoder(read_golden("decodecorpus", "z000088.zst"))
    out = s.read_to_end()
    assert hashlib.sha256(out).hexdigest() == manifest["corpus"]["z000088.zst"]["sha256"]
    s2 = oracle.StreamingDecoder(read_golden("decodecorpus", "z000068.zst"), decoder=s.into_frame_decoder())
    assert hashlib.sha256(s2.read_to_end()).hexdigest() == manifest["corpus"]["z000068.zst"]["sha256"]


def test_api_incremental_read(oracle):
    """tests/mod.rs:382-404."""
    data = read_golden("decodecorpus", "abc.txt.zst")
    d = oracle.FrameDecoder()
    r = d.reset(data)
    rest = r.src.read()
    _, out = d.decode_from_to(rest, 3)
    assert out == b"abc" and d.is_finished()
    assert d.read(3) == b"def"


def test_api_decode_all(oracle, manifest):
    """tests/mod.rs:490-574: skippable frames, too small / too large output, truncated input."""
    def skip(n):
        return (0x184D2A50).to_bytes(4, "little") + n.to_bytes(4, "little") + bytes(n)
    a, b = read_golden("decodecorpus", "z000089.zst"), read_golden("decodecorpus", "z000090.zst")
    inp = skip(300) + a + skip(400) + b + skip(500)
    total = manifest["corpus"]["z000089.zst"]["size"] + manifest["corpus"]["z000090.zst"]["size"]
    d = oracle.FrameDecoder()
    out = d.decode_all(inp, total)
    assert len(out) == total
    names = oracle.error_names()
    with pytest.raises(oracle.OracleError) as e:
        d.decode_all(inp, total - 1)
    assert names[e.value.code] == "ZO_ERR_TARGET_TOO_SMALL"
    assert d.decode_all(inp, total + 1) == out
    with pytest.raises(oracle.OracleError) as e:
        d.decode_all(inp[:-600], total)
    assert e.value.stage in (3, 4, 5, 6) or names[e.value.code] in ("ZO_ERR_BLOCK_CONTENT_READ", "ZO_ERR_BLOCK_BODY_READ")
    with pytest.raises(oracle.OracleError) as e:
        d.decode_all(inp[:-1], total)
    assert names[e.value.code] == "ZO_ERR_FAILED_TO_SKIP_FRAME"


def test_against_libzstd_on_synthetic(oracle):
    """Secondary oracle: decode(libzstd level-3 output) == input (fuzz/fuzz_targets/interop.rs:55-65), incl. chained
    blocks, a raw-content dictionary and mixed Raw/RLE/Compressed blocks."""
    import datagen as G
    text = G.gen_text(600_000, 5)
    f = G.compress(text, window_log=17)
    out, d = oracle.decode_frame(f)
    assert out == text.tobytes() and d.get_checksum_from_data() == d.get_calculated_checksum()
    assert G.decompress(f, len(text)) == out
    mix = G.gen_silesia_mix(1 << 20, 0xC40000)
    f = G.compress(mix)
    assert oracle.decode_frame(f)[0] == mix.tobytes()
    dic = G.gen_text(112640, 0xD1C7)
    piece = dic[1000:1400].tobytes() + G.gen_text(300, 9).tobytes() + dic[50000:50700].tobytes()
    f = G.compress(piece, raw_dict=dic)
    assert oracle.decode_frame(f, raw_dict=dic.tobytes())[0] == piece
    assert G.decompress(f, len(piece), raw_dict=dic) == piece
