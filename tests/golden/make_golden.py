#!/usr/bin/env python3
"""Generate tests/golden/ from the reference's own golden vectors.  usage: make_golden.py <zstd-rs checkout>

The reference (KillingSpark/zstd-rs @ eb7e03cc) is Rust and cannot be executed here, so the vectors are the
ones its own tests assert on (SURVEY.md section 8c):
  * ruzstd/decodecorpus_files/*.zst + originals   (tests/decode_corpus.rs)
  * ruzstd/dict_tests/{dictionary,files/*}        (tests/dict_test.rs)
  * ruzstd/test_fixtures/*.zst                    (tests/mod.rs:576-741; plaintexts generated in code)
  * ruzstd/fuzz/artifacts/*/*                     (tests/fuzz_regressions.rs, fse/mod.rs, huff0/mod.rs)
Compressed inputs are copied verbatim (they are test DATA, not source); expected plaintexts are recorded as
size + SHA-256 + XXH64-low32 in manifest.json so the repo stays small, and byte windows of every decode-corpus
original (first and last 64 bytes, four seeded 32-byte windows in between) go to decodecorpus_originals.npz.
Every test reads tests/golden/ only; the reference checkout is needed to regenerate it, not to run the tests.
"""
import hashlib, json, os, shutil, sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))


def sha(b):
    return hashlib.sha256(b).hexdigest()


def original_windows(orig, rng):
    """(offset, length) of the stored windows of one original: all of it when short, else head, tail and 4 seeded windows."""
    if len(orig) <= 256:
        return [(0, len(orig))]
    mid = sorted(int(x) for x in rng.integers(64, len(orig) - 96, 4))
    return [(0, 64)] + [(o, 32) for o in mid] + [(len(orig) - 64, 64)]


def main(ref):
    from oracle.oracle import xxh64
    REF = os.path.join(ref, "ruzstd")
    man = {"source": "KillingSpark/zstd-rs eb7e03cc1b15705b94b93249ff7b05c4fc2c98b3", "corpus": {}, "dict": {}, "fixtures": {}, "fuzz": {}}
    # corpus
    dst = os.path.join(HERE, "decodecorpus"); os.makedirs(dst, exist_ok=True)
    rng = np.random.Generator(np.random.PCG64(0xD0C0))
    names, sizes, win_file, win_off, win_len, vals = [], [], [], [], [], []
    for f in sorted(os.listdir(f"{REF}/decodecorpus_files")):
        if not f.endswith(".zst"):
            continue
        shutil.copyfile(f"{REF}/decodecorpus_files/{f}", f"{dst}/{f}")
        orig = open(f"{REF}/decodecorpus_files/{f[:-4]}", "rb").read()
        man["corpus"][f] = {"size": len(orig), "sha256": sha(orig), "xxh64_low32": xxh64(orig) & 0xFFFFFFFF,
                            "compressed_size": os.path.getsize(f"{dst}/{f}")}
        for o, n in original_windows(orig, rng):
            win_file.append(len(names)); win_off.append(o); win_len.append(n); vals.append(np.frombuffer(orig[o:o + n], np.uint8))
        names.append(f); sizes.append(len(orig))
    np.savez_compressed(os.path.join(HERE, "decodecorpus_originals.npz"), name=np.array(names), size=np.array(sizes, np.uint64),
                        win_file=np.array(win_file, np.uint32), win_off=np.array(win_off, np.uint64),
                        win_len=np.array(win_len, np.uint32), val=np.concatenate(vals))
    # dict tests
    dst = os.path.join(HERE, "dict_tests", "files"); os.makedirs(dst, exist_ok=True)
    shutil.copyfile(f"{REF}/dict_tests/dictionary", os.path.join(HERE, "dict_tests", "dictionary"))
    for f in sorted(os.listdir(f"{REF}/dict_tests/files")):
        if not f.endswith(".zst"):
            continue
        shutil.copyfile(f"{REF}/dict_tests/files/{f}", f"{dst}/{f}")
        orig = open(f"{REF}/dict_tests/files/{f[:-4]}", "rb").read()
        man["dict"][f] = {"size": len(orig), "sha256": sha(orig), "compressed_size": os.path.getsize(f"{dst}/{f}")}
    # window fixtures: plaintexts are generated in code by the reference tests (tests/mod.rs:582-595)
    dst = os.path.join(HERE, "test_fixtures"); os.makedirs(dst, exist_ok=True)
    fox = b"The quick brown fox jumps over the lazy dog.\n" * 4096
    sphinx = b"Sphinx of black quartz, judge my vow.\n" * 4096
    abc = b"abcdefghijklmnopqrstuvwxyz"
    plain = {"window_128mib.zst": fox, "window_256mib.zst": fox, "window_8mib.zst": sphinx, "abc.txt.zst": abc}
    for f in sorted(os.listdir(f"{REF}/test_fixtures")):
        shutil.copyfile(f"{REF}/test_fixtures/{f}", f"{dst}/{f}")
        p = plain[f]
        man["fixtures"][f] = {"size": len(p), "sha256": sha(p)}
    # fuzz artifacts
    for sub in sorted(os.listdir(f"{REF}/fuzz/artifacts")):
        dst = os.path.join(HERE, "fuzz", sub); os.makedirs(dst, exist_ok=True)
        man["fuzz"][sub] = []
        for f in sorted(os.listdir(f"{REF}/fuzz/artifacts/{sub}")):
            shutil.copyfile(f"{REF}/fuzz/artifacts/{sub}/{f}", f"{dst}/{f}")
            man["fuzz"][sub].append(f)
    json.dump(man, open(os.path.join(HERE, "manifest.json"), "w"), indent=1, sort_keys=True)
    print("corpus", len(man["corpus"]), "dict", len(man["dict"]), "fixtures", len(man["fixtures"]),
          "fuzz", sum(len(v) for v in man["fuzz"].values()))


if __name__ == "__main__":
    main(sys.argv[1])
