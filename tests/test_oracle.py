"""Pin the oracle (oracle/mzoracle.c) before anything trusts it.

Checked against (a) the reference's golden fixtures (seed-corpus DEFLATE/STORE entries with header CRCs,
random.bin CRC), (b) streams and CRCs produced by the reference itself (oracle/_ref, committed as
tests/golden/golden_vectors.json by make_golden.py), (c) CPython's zlib module (system zlib 1.3) as an
independent implementation, (d) the reference's outputs for larger seeded inputs (tests/golden/reference_outputs.json).
"""
import zlib

import pytest

import datagen
import refshim


def _payload(ent):
    if "payload_hex" in ent:
        return bytes.fromhex(ent["payload_hex"])
    return bytes([ent["fill_byte"]]) * ent["csize"]


def test_crc_known_answers(orc, golden):
    assert orc.crc32(0, b"") == 0
    assert orc.crc32(0, b"123456789") == 0xCBF43926
    assert orc.crc32(orc.crc32(0, b"1234"), b"56789") == 0xCBF43926
    seen = 0
    for v in golden["crc"]:
        if v["input"] == "ascii_123456789":
            assert v["crc32"] == 0xCBF43926
            seen += 1
        if v["input"].startswith("reference:test/random.bin"):
            assert v["crc32"] == 0xA85D40DC
            seen += 1
    assert seen == 2


def test_crc_foreign_store_entries(orc, golden):
    n = 0
    for ent in golden["foreign"]:
        if ent["method"] == 0:
            assert orc.crc32(0, _payload(ent)) == ent["crc32"], ent["name"]
            n += 1
    assert n >= 5


def test_inflate_foreign_deflate_entries(orc, golden):
    n = 0
    for ent in golden["foreign"]:
        if ent["method"] != 8:
            continue
        comp = _payload(ent)
        err, out, cons = orc.inflate(comp + b"\xAA" * 7, ent["size"] + 16)
        assert err == 0, (ent["zip"], ent["name"], err)
        assert cons == len(comp)
        assert len(out) == ent["size"]
        assert orc.crc32(0, out) == ent["crc32"]
        assert zlib.decompress(comp, -15) == out
        n += 1
    assert n >= 10


def test_inflate_reference_streams(orc, golden):
    for v in golden["refrun"]:
        comp = bytes.fromhex(v["stream_hex"])
        err, out, cons = orc.inflate(comp, v["size"] + 8, v["window_bits"])
        assert err == 0, v["input"]
        assert cons == len(comp)
        assert len(out) == v["size"] and orc.crc32(0, out) == v["crc32"]


def test_reference_boundary_bytes(golden):
    """Exact bytes the survey observed from mz_strm_zlib (SURVEY.md 8c table)."""
    by = {(v["input"], v["level"], v["window_bits"]): bytes.fromhex(v["stream_hex"]) for v in golden["refrun"]}
    assert by[("empty", 6, -15)] == bytes.fromhex("0300")
    assert by[("empty", 6, 31)] == bytes.fromhex("1f8b0800000000000003" "0300" "00000000" "00000000")
    assert by[("a", 6, -15)] == bytes.fromhex("4b0400")
    assert by[("hello", 6, 31)] == bytes.fromhex("1f8b0800000000000003cb48cdc9c9070086a6103605000000")
    assert by[("hello", 1, 31)][8] == 4  # XFL for level 1
    assert by[("hello", 0, -15)] == bytes.fromhex("010500faff") + b"hello"


def test_inflate_errors(orc, golden):
    v = next(v for v in golden["refrun"] if v["input"] == "text_3k" and v["level"] == 6 and v["window_bits"] == 31)
    comp = bytearray(bytes.fromhex(v["stream_hex"]))
    err, _, _ = orc.inflate(bytes(comp[:len(comp) // 2]), v["size"] + 8, 31)
    assert err == -5  # truncated -> BUF_ERROR (mz_strm_zlib behaviour, SURVEY 8c)
    bad = bytearray(comp)
    bad[-8] ^= 0xFF
    err, _, _ = orc.inflate(bytes(bad), v["size"] + 8, 31)
    assert err == -3  # wrong trailer CRC -> DATA_ERROR
    raw = next(v for v in golden["refrun"] if v["input"] == "text_3k" and v["level"] == 6 and v["window_bits"] == -15)
    err, _, _ = orc.inflate(bytes.fromhex(raw["stream_hex"]), v["size"] + 8, 31)
    assert err == -3  # raw fed to a gzip reader
    err, _, _ = orc.inflate(bytes.fromhex(raw["stream_hex"]), 100, -15)
    assert err == -5  # short output


@pytest.mark.parametrize("n,seed", [(0, 1), (1, 2), (17, 3), (4095, 4), (65536, 5), (300000, 6)])
def test_crc_vs_system_zlib(orc, n, seed):
    data = datagen.random_bytes(n, seed)
    assert orc.crc32(0, data) == zlib.crc32(data)
    k = n // 3
    assert orc.crc32(orc.crc32(0, data[:k]), data[k:]) == zlib.crc32(data)
    assert orc.crc32_combine(zlib.crc32(data[:k]), zlib.crc32(data[k:]), n - k) == zlib.crc32(data)


def test_crc_combine_large_lengths(orc):
    a, b, c = 0x12345678, 0x9ABCDEF0, 0x0F1E2D3C
    for ln in (1, 2, 3, 255, 65536, (1 << 31) + 7, (1 << 34) + 12345):
        # associativity: combine(a, combine(b, c, l2), l1 + l2) == combine(combine(a, b, l1), c, l2)
        l1, l2 = ln, (ln * 7 + 3) % (1 << 33)
        lhs = orc.crc32_combine(a, orc.crc32_combine(b, c, l2), l1 + l2)
        rhs = orc.crc32_combine(orc.crc32_combine(a, b, l1), c, l2)
        assert lhs == rhs


@pytest.mark.parametrize("kind", ["text", "records", "random", "zeros", "mixed"])
@pytest.mark.parametrize("level", [0, 1, 6])
def test_oracle_deflate_roundtrip(orc, kind, level):
    n = 150000
    data = {"text": datagen.text_like(n, 21), "records": datagen.binary_records(n, 22),
            "random": datagen.random_bytes(n, 23), "zeros": bytes(n), "mixed": datagen.mixed(n, 24)}[kind]
    for wb in (-15, 31, 15):
        comp = orc.deflate(data, level, wb)
        assert zlib.decompress(comp, wb) == data  # independent decoder
        err, out, cons = orc.inflate(comp, n + 8, wb)
        assert err == 0 and out == data and cons == len(comp)


def test_oracle_matches_live_reference(orc):
    """The restatement and the reference agree on fresh inputs, both directions (the reference's CRCs and streams pinned in
    tests/golden/reference_outputs.json; its reader is zlib's inflate)."""
    pinned = refshim.reference_outputs()["oracle"]
    assert [(e["seed"], e["n"]) for e in pinned] == [(31, 0), (32, 1), (33, 5000), (34, 200000)]
    for e in pinned:
        n = e["n"]
        data = datagen.mixed(n, e["seed"]) if n else b""
        assert e["crc32"] == orc.crc32(0, data)
        assert [(s["level"], s["window_bits"]) for s in e["streams"]] == [(1, -15), (6, 31), (9, -15)]
        for s in e["streams"]:
            level, wb = s["level"], s["window_bits"]
            comp = refshim.zlib_stream(data, level, wb)
            assert refshim.is_reference_stream(comp, s), (n, level, wb)
            err, out, cons = orc.inflate(comp, n + 8, wb)
            assert err == 0 and out == data and cons == len(comp)
            mine = orc.deflate(data, level, wb)
            assert refshim.zlib_read(mine, wb) == (data, len(mine), True)


def test_block_walker(orc, golden):
    v = next(v for v in golden["refrun"] if v["input"] == "run_a_70k" and v["level"] == 0)
    blocks, prod = orc.blocks(bytes.fromhex(v["stream_hex"]), -15)
    assert prod == 70000 and len(blocks) == 3 and all(b[2] == 0 for b in blocks) and blocks[-1][3] == 1
