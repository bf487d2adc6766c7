#!/usr/bin/env python3
"""Generate tests/golden/golden_vectors.json from the reference tree and from the reference run here.

Run in the build container (needs /root/reference and oracle/_ref/libmzref.so); the GPU box only
reads the committed JSON.  Two families of vectors:

1. ``foreign``: every DEFLATE (method 8) and STORE (method 0) entry of the reference's fuzz seed
   corpus (test/fuzz/unzip_fuzzer_seed_corpus/*.zip) -- the only known-answer vectors the reference
   holds for inflate + CRC-32 (SURVEY.md section 8c).  We keep the raw compressed payload, the CRC-32
   and the sizes recorded in the zip headers by the third-party tools that made them.
2. ``refrun``: streams produced HERE by the reference's own mz_stream_zlib (mz_strm_zlib.c) over
   system zlib 1.3 at several levels / window_bits, for deterministic seeded inputs, plus the CRC
   returned by the reference's mz_crypt_crc32_update (mz_crypt.c:35).  Includes the boundary cases
   the survey observed (empty input, "a", "hello" gzip, level 0 stored).

It also writes ``reference_outputs.json``: the reference's outputs for the larger seeded inputs of the tests that
compare with it, pinned by CRC-32, length and SHA-256 so that those tests need no reference build.
"""
import ctypes
import hashlib
import json
import os
import struct
import sys
import zipfile
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("MZ_REFERENCE", "/root/reference")
sys.path.insert(0, os.path.join(ROOT, "tests"))


def corpus_entries():
    out = []
    cdir = os.path.join(REF, "test/fuzz/unzip_fuzzer_seed_corpus")
    for name in sorted(os.listdir(cdir)):
        path = os.path.join(cdir, name)
        try:
            zf = zipfile.ZipFile(path)
        except Exception:
            continue
        raw = open(path, "rb").read()
        for zi in zf.infolist():
            if zi.compress_type not in (0, 8) or zi.flag_bits & 1:
                continue
            off = zi.header_offset
            if raw[off:off + 4] != b"PK\x03\x04":
                continue
            nlen, xlen = struct.unpack("<HH", raw[off + 26:off + 30])
            start = off + 30 + nlen + xlen
            payload = raw[start:start + zi.compress_size]
            if len(payload) != zi.compress_size:
                continue
            ent = {
                "zip": name, "name": zi.filename, "method": zi.compress_type,
                "crc32": zi.CRC, "size": zi.file_size, "csize": zi.compress_size,
            }
            if zi.compress_type == 8:
                data = zlib.decompress(payload, -15)
                assert zlib.crc32(data) == zi.CRC and len(data) == zi.file_size
                ent["payload_hex"] = payload.hex()
            else:
                assert zlib.crc32(payload) == zi.CRC
                if len(payload) <= 4096:
                    ent["payload_hex"] = payload.hex()
                elif len(set(payload)) == 1:
                    ent["fill_byte"] = payload[0]
                else:
                    continue
            out.append(ent)
    return out


def seeded_inputs():
    from datagen import text_like, binary_records
    rng = np.random.default_rng(7)
    return {
        "empty": b"",
        "a": b"a",
        "hello": b"hello",
        "text_3k": text_like(3000, seed=11),
        "text_20k": text_like(20000, seed=12),
        "records_8k": binary_records(8192, seed=13),
        "random_2k": rng.integers(0, 256, 2048, dtype=np.uint8).tobytes(),
        "zeros_5k": bytes(5000),
        "run_a_70k": b"A" * 70000,
    }


def _digest(stream):
    return {"size": len(stream), "sha256": hashlib.sha256(stream).hexdigest()}


def reference_outputs(ref):
    """What the reference's own mz_stream_zlib / mz_crypt_crc32_update return for the seeded inputs of the tests that compare
    with it (tests/test_oracle.py, tests/test_gpu_parity.py, tests/test_gpu_configs.py). Streams are pinned by length and
    SHA-256: the reference's writer is zlib's deflate, so the tests rebuild each stream with CPython's zlib, prove it is the
    reference's by the digest, and then feed it to the code under test."""
    from datagen import mixed
    import textgen
    out = {"oracle": [], "parity_crc": [], "c3_member": None}
    for seed, n in ((31, 0), (32, 1), (33, 5000), (34, 200000)):
        data = mixed(n, seed) if n else b""
        streams = []
        for level, wb in ((1, -15), (6, 31), (9, -15)):
            comp = ref.zlib_compress(data, level, wb)
            streams.append(dict(level=level, window_bits=wb, **_digest(comp)))
        out["oracle"].append({"seed": seed, "n": n, "crc32": ref.crc32(0, data), "streams": streams})
    for wb in (-15, 31):
        for level in (1, 6):
            seed = wb + level + 50
            out["parity_crc"].append({"seed": seed, "n": 700000, "crc32": ref.crc32(0, mixed(700000, seed))})
    n = 128 << 20
    text = textgen.host(n, seed=7)
    comp = ref.zlib_compress(text, level=6, window_bits=31, write_size=1 << 20)
    out["c3_member"] = dict(text_seed=7, n=n, level=6, window_bits=31, crc32=ref.crc32(0, text), **_digest(comp))
    return out


def main():
    import refshim
    ref = refshim.RefLib()
    json.dump(reference_outputs(ref), open(os.path.join(HERE, "reference_outputs.json"), "w"), indent=1)
    vec = {"foreign": corpus_entries(), "refrun": [], "crc": []}
    inputs = seeded_inputs()
    for key, data in inputs.items():
        for level, wbits in ((1, -15), (6, -15), (9, -15), (6, 31), (0, -15), (1, 31)):
            if len(data) > 30000 and level == 9:
                continue
            comp = ref.zlib_compress(data, level=level, window_bits=wbits, write_size=16384)
            assert ref.zlib_decompress(comp, window_bits=wbits) == data
            vec["refrun"].append({
                "input": key, "level": level, "window_bits": wbits,
                "stream_hex": comp.hex(), "size": len(data), "crc32": ref.crc32(0, data),
            })
    for key, data in inputs.items():
        vec["crc"].append({"input": key, "size": len(data), "crc32": ref.crc32(0, data)})
    vec["crc"].append({"input": "ascii_123456789", "size": 9, "crc32": ref.crc32(0, b"123456789")})
    rb = open(os.path.join(REF, "test/random.bin"), "rb").read()
    vec["crc"].append({"input": "reference:test/random.bin", "size": len(rb), "crc32": ref.crc32(0, rb),
                       "note": "file not committed; value pinned, SURVEY 8c says a85d40dc"})
    json.dump(vec, open(os.path.join(HERE, "golden_vectors.json"), "w"), indent=1)
    print("foreign", len(vec["foreign"]), "refrun", len(vec["refrun"]), "crc", len(vec["crc"]))


if __name__ == "__main__":
    main()
