"""GPU parity tests (pytest -m gpu): the CUDA path, called through the C ABI, against the oracle.

Bar (bit-exact, integer/byte work): every stream we write is inflated by the oracle (oracle/mzoracle.c) and
-- when it travelled -- by the reference's own mz_stream_zlib_read to exactly the input; every stream the
reference / third parties wrote is inflated by us to exactly their output; every CRC equals the
reference's.  Compressed bytes are not compared with zlib's (SURVEY.md section 4: the reference's tests never do).
"""
import ctypes as C
import os
import zlib

import pytest

import datagen
import refshim

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cu(built):
    import cuharness
    p = cuharness.pkg()
    lib = p.load()
    err = lib.mz_cuda_init()
    assert err == 0, "mz_cuda_init failed: %d %s" % (err, lib.mz_cuda_last_error())
    return p, lib, cuharness.TestLib()


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return torch


def _dev(torch, data):
    import numpy as np
    t = torch.from_numpy(np.frombuffer(bytes(data) if len(data) else b"\0", dtype=np.uint8).copy()).cuda()
    return t


INPUTS = {
    "text": lambda n, s: datagen.text_like(n, s),
    "records": lambda n, s: datagen.binary_records(n, s),
    "random": lambda n, s: datagen.random_bytes(n, s),
    "zeros": lambda n, s: bytes(n),
    "mixed": lambda n, s: datagen.mixed(n, s),
    "abc": lambda n, s: (b"abcabcabd" * (n // 9 + 1))[:n],
}


# ---- K1: CRC-32 -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 15, 16, 17, 511, 512, 513, 4096, 65535, 65536, 65537, 1 << 20, (1 << 24) + 3])
def test_crc_device_vs_oracle(cu, torch_cuda, orc, n):
    p, lib, _ = cu
    data = datagen.random_bytes(n, n + 1)
    t = _dev(torch_cuda, data)
    for mis in (0, 1, 5):
        if n < mis:
            continue
        view = t[mis:]
        assert p.crc32_device(view, n - mis) == orc.crc32(0, data[mis:])
    k = n // 3
    assert p.crc32_device(t[k:], n - k, value=orc.crc32(0, data[:k])) == orc.crc32(0, data)  # chaining


def test_crc_known_answers_and_golden(cu, torch_cuda, golden):
    p, lib, _ = cu
    assert p.crc32_device(_dev(torch_cuda, b"123456789"), 9) == 0xCBF43926
    for ent in golden["foreign"]:
        if ent["method"] == 0:
            payload = bytes.fromhex(ent["payload_hex"]) if "payload_hex" in ent else bytes([ent["fill_byte"]]) * ent["csize"]
            assert p.crc32_device(_dev(torch_cuda, payload), len(payload)) == ent["crc32"], ent["name"]


def test_crc_per_segment_and_combine(cu, torch_cuda, orc):
    p, lib, _ = cu
    n = 5 * 65536 + 777
    data = datagen.mixed(n, 3)
    t = _dev(torch_cuda, data)
    nseg = (n + 65535) // 65536
    res = torch_cuda.empty(nseg, dtype=torch_cuda.int32, device="cuda")
    crc = torch_cuda.empty(nseg, dtype=torch_cuda.int32, device="cuda")
    p.check(lib.mz_cuda_crc32_segments(t.data_ptr(), n, 65536, None, None, nseg, res.data_ptr(), crc.data_ptr(), None))
    torch_cuda.cuda.synchronize()
    crcs = [int(x) & 0xFFFFFFFF for x in crc.cpu().tolist()]
    acc = 0
    for i, c in enumerate(crcs):
        seg = data[i * 65536:(i + 1) * 65536]
        assert c == orc.crc32(0, seg)
        acc = lib.mz_cuda_crc32_combine(acc, c, len(seg)) if i else c
    assert acc == orc.crc32(0, data)  # checksum of checksums == checksum of the whole
    assert lib.mz_cuda_crc32_combine(0x12345678, 0x9ABCDEF0, (1 << 34) + 5) == orc.crc32_combine(0x12345678, 0x9ABCDEF0, (1 << 34) + 5)


def test_crc_replacement_symbol(cu, orc, monkeypatch):
    """mz_crypt_crc32_update: same contract as mz_crypt.c:35 on both sides of the size threshold."""
    p, lib, _ = cu
    data = datagen.mixed(3 << 20, 9)
    buf = C.create_string_buffer(data, len(data))
    assert lib.mz_crypt_crc32_update(0, buf, 0) == 0
    assert lib.mz_crypt_crc32_update(0x1234, buf, 0) == 0x1234
    assert lib.mz_crypt_crc32_update(0, buf, 9) == orc.crc32(0, data[:9])                     # host table path
    assert lib.mz_crypt_crc32_update(0, buf, len(data)) == orc.crc32(0, data)               # GPU path
    half = len(data) // 2
    v = lib.mz_crypt_crc32_update(0, buf, half)
    v = lib.mz_crypt_crc32_update(v, C.byref(buf, half), len(data) - half)
    assert v == orc.crc32(0, data)                                                           # chaining across calls


# ---- K2+K3+K4: device batch API ---------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", sorted(INPUTS))
@pytest.mark.parametrize("level", [0, 1, 6])
def test_deflate_batch_roundtrip(cu, torch_cuda, orc, kind, level):
    p, lib, _ = cu
    for n in (0, 1, 5, 33, 32768, 65535, 65536, 65537, 300001):
        data = INPUTS[kind](n, n + level)
        t = _dev(torch_cuda, data)
        b = p.DeflateBatch(max(n, 1))
        k = b.compress(t, n, level=level, final=True)
        joined, crc = b.result(k)
        comp = bytes(joined.cpu().numpy().tobytes())
        err, out, cons = orc.inflate(comp, n + 8)
        assert err == 0 and out == data and cons == len(comp), (kind, level, n, err)
        assert zlib.decompress(comp, -15) == data
        if n:
            assert crc == orc.crc32(0, data)


def test_deflate_history_variant_on_gpu(cu, torch_cuda, orc):
    """levels 6-9 = the kernel's history variant (208 KiB of shared memory, one CTA per SM): independent chunks and one-stream mode
    (MZ_CUDA_FLAG_DICT); same checks as on the emulator (tests/test_emu_kernels.py), bigger inputs"""
    p, lib, _ = cu
    import datagen
    for data in (datagen.text_like(3_000_001, 31), datagen.mixed(2_000_000, 32), bytes(1_000_000), datagen.random_bytes(700_000, 33),
                 (datagen.random_bytes(30_000, 34) * 40)[:1_100_000]):
        n = len(data)
        t = _dev(torch_cuda, data)
        sizes = {}
        for level, one in ((3, False), (6, False), (6, True), (9, True)):
            b = p.DeflateBatch(n)
            k = b.compress(t, n, level=level, final=True, one_stream=one)
            joined, crc = b.result(k)
            comp = bytes(joined.cpu().numpy().tobytes())
            assert zlib.decompress(comp, -15) == data, (n, level, one)
            err, out, cons = orc.inflate(comp, n + 8)
            assert err == 0 and out == data and cons == len(comp)
            assert crc == orc.crc32(0, data)
            sizes[(level, one)] = len(comp)
        if data[:64] != bytes(64):
            assert sizes[(6, True)] <= sizes[(6, False)] <= sizes[(3, False)] * 1.002, sizes
    assert sizes[(6, True)] < 0.1 * n  # the 30 000-byte period is only visible through the history


def test_deflate_runs_and_near_sources_on_gpu(cu, torch_cuda, orc):
    """same inputs as tests/test_emu_kernels.py::test_emu_deflate_runs_and_near_sources, on the device"""
    p, lib, _ = cu
    import datagen
    traps = datagen.near_period_traps()
    cases = [traps, bytes(2_000_000), (b"abc" * 700_000)[:2_000_001], b"".join(bytes([i & 255]) * (5 + 13 * i % 700) for i in range(3000)),
             b"".join(datagen.random_bytes(37, i) + bytes(3000 + 17 * i) for i in range(200)), traps[:32768] + bytes(40_000) + traps[:20_000]]
    for data in cases:
        n = len(data)
        t = _dev(torch_cuda, data)
        for level, one in ((1, False), (3, False), (6, False), (9, True)):
            b = p.DeflateBatch(n)
            k = b.compress(t, n, level=level, final=True, one_stream=one)
            joined, crc = b.result(k)
            comp = bytes(joined.cpu().numpy().tobytes())
            assert zlib.decompress(comp, -15) == data, (n, level, one)
            assert crc == orc.crc32(0, data)
            if data[:4096] == bytes(4096) and data[-4096:] == bytes(4096):
                assert len(comp) < 0.006 * n  # zeros: ~130 bytes per 32 KiB (zlib level 1: 0.0044)


def test_deflate_empty_stream_bytes(cu, torch_cuda):
    p, lib, _ = cu
    b = p.DeflateBatch(1)
    k = b.compress(_dev(torch_cuda, b""), 0, level=6, final=True)
    joined, _ = b.result(k)
    assert bytes(joined.cpu().numpy().tobytes()) == bytes.fromhex("0300")  # what mz_strm_zlib emits (SURVEY 8c)


def test_deflate_nonfinal_chunks_join(cu, torch_cuda, orc):
    """Non-final batches end with a sync marker; concatenating batches gives one valid stream."""
    p, lib, _ = cu
    parts = [datagen.text_like(100000, 1), datagen.random_bytes(70000, 2), datagen.text_like(5, 3)]
    comp = b""
    for i, d in enumerate(parts):
        b = p.DeflateBatch(len(d))
        k = b.compress(_dev(torch_cuda, d), len(d), level=1, final=(i == len(parts) - 1))
        joined, _ = b.result(k)
        comp += bytes(joined.cpu().numpy().tobytes())
    whole = b"".join(parts)
    err, out, cons = orc.inflate(comp, len(whole) + 8)
    assert err == 0 and out == whole and cons == len(comp)


def test_deflate_entries_api(cu, torch_cuda, orc):
    """Explicit per-chunk offsets/lengths/flags (zip entries of ragged size, config C4 shape)."""
    p, lib, _ = cu
    import numpy as np
    torch = torch_cuda
    sizes = [65536, 1, 0, 4097, 65535, 12345, 65536, 333]
    blobs = [datagen.mixed(s, 100 + i) for i, s in enumerate(sizes)]
    offs, pos = [], 0
    for s in sizes:
        offs.append(pos)
        pos += s + 3  # deliberately unaligned
    big = bytearray(pos + 16)
    for o, bl in zip(offs, blobs):
        big[o:o + len(bl)] = bl
    t = _dev(torch, bytes(big))
    d_off = torch.tensor(offs, dtype=torch.int64, device="cuda")
    d_len = torch.tensor(sizes, dtype=torch.int32, device="cuda")
    d_flags = torch.ones(len(sizes), dtype=torch.uint8, device="cuda")  # every entry is its own final stream
    stride = int(lib.mz_cuda_deflate_slot_bound(65536))
    slots = torch.empty(len(sizes) * stride, dtype=torch.uint8, device="cuda")
    out_len = torch.empty(len(sizes), dtype=torch.int32, device="cuda")
    p.check(lib.mz_cuda_deflate_chunks(t.data_ptr(), 0, 0, d_off.data_ptr(), d_len.data_ptr(), d_flags.data_ptr(), len(sizes), 0, 6,
                                       slots.data_ptr(), stride, out_len.data_ptr(), None))
    res = torch.empty(len(sizes), dtype=torch.int32, device="cuda")
    crc = torch.empty(len(sizes), dtype=torch.int32, device="cuda")
    p.check(lib.mz_cuda_crc32_segments(t.data_ptr(), 0, 0, d_off.data_ptr(), d_len.data_ptr(), len(sizes), res.data_ptr(), crc.data_ptr(), None))
    torch.cuda.synchronize()
    lens = out_len.cpu().tolist()
    raw = slots.cpu().numpy()
    for i, bl in enumerate(blobs):
        comp = raw[i * stride:i * stride + lens[i]].tobytes()
        err, out, cons = orc.inflate(comp, len(bl) + 8)
        assert err == 0 and out == bl and cons == len(comp), i
        assert (int(crc[i]) & 0xFFFFFFFF) == orc.crc32(0, bl)


# ---- the vtbl stream: write path (test_stream_compress.cc flow) ------------------------------------------------
@pytest.mark.parametrize("wb", [-15, 31, 15])
@pytest.mark.parametrize("level", [-1, 0, 1, 9])
def test_stream_write_roundtrip(cu, orc, wb, level):
    p, lib, tl = cu
    for n, ws in ((0, 16384), (1, 16384), (877, 16384), (200000, 16384), (200000, 65535), (3 << 20, 1 << 20)):
        data = datagen.mixed(n, n + 7) if n else b""
        comp, info = tl.compress(lib.mz_stream_cuda_create, data, level=level, window_bits=wb, write_size=ws)
        assert info["open"] == 0 and info["wrote"] == n and info["close"] == 0
        assert info["total_in"] == n                       # test_stream_compress.cc:78-79
        assert info["total_out"] == len(comp) == info["sink_tell"]  # :81-82
        assert info["is_open_after_close"] == refshim.MZ_OPEN_ERROR  # SURVEY 8c: props readable, is_open -111
        err, out, cons = orc.inflate(comp, n + 8, wb)
        assert err == 0 and out == data and cons == len(comp), (wb, level, n, err)
        assert zlib.decompress(comp, wb) == data


def test_stream_write_gzip_framing_bytes(cu):
    p, lib, tl = cu
    comp, _ = tl.compress(lib.mz_stream_cuda_create, b"", level=6, window_bits=31)
    assert comp == bytes.fromhex("1f8b0800000000000003" "0300" "00000000" "00000000")  # == the reference, SURVEY 8c
    comp, _ = tl.compress(lib.mz_stream_cuda_create, b"hello", level=1, window_bits=31, open_before_base=True)
    assert comp[:10] == bytes.fromhex("1f8b0800000000000403") and comp[-8:] == bytes.fromhex("86a6103605000000")
    comp, _ = tl.compress(lib.mz_stream_cuda_create, b"hello", level=9, window_bits=31)
    assert comp[8] == 2
    comp, _ = tl.compress(lib.mz_stream_cuda_create, b"hello", level=0, window_bits=-15)
    assert comp == bytes.fromhex("010500faff") + b"hello"  # == the reference at level 0


def test_stream_write_multi_batch(cu, orc, monkeypatch):
    """Small staging batches: several non-final batches + a final one must still be one valid member."""
    p, lib, tl = cu
    monkeypatch.setenv("MZ_CUDA_BATCH_KB", "128")
    data = datagen.mixed(128 * 1024 * 3, 5)  # exact multiple: close() must add an empty final block
    for wb in (-15, 31):
        comp, info = tl.compress(lib.mz_stream_cuda_create, data, level=1, window_bits=wb, write_size=65535)
        err, out, cons = orc.inflate(comp, len(data) + 8, wb)
        assert err == 0 and out == data and cons == len(comp) == info["total_out"]
    data = data + b"tail"
    comp, info = tl.compress(lib.mz_stream_cuda_create, data, level=6, window_bits=31, write_size=16384)
    assert zlib.decompress(comp, 31) == data


def test_stream_open_validation(cu):
    p, lib, tl = cu
    for level, wb in ((10, -15), (200, -15), (6, -7), (6, 16), (6, 40)):
        comp, info = tl.compress(lib.mz_stream_cuda_create, b"x", level=level, window_bits=wb)
        assert comp is None and info["open"] == refshim.MZ_OPEN_ERROR, (level, wb)
    s = lib.mz_stream_cuda_create()
    v = C.c_int64(0)
    assert lib.mz_stream_cuda_get_prop_int64(s, 99, C.byref(v)) == refshim.MZ_EXIST_ERROR
    assert lib.mz_stream_cuda_set_prop_int64(s, 99, 1) == refshim.MZ_EXIST_ERROR
    assert lib.mz_stream_cuda_get_prop_int64(s, refshim.PROP_COMPRESS_WINDOW, C.byref(v)) == 0 and v.value == -15
    assert lib.mz_stream_cuda_get_prop_int64(s, refshim.PROP_HEADER_SIZE, C.byref(v)) == 0 and v.value == 0
    assert lib.mz_stream_cuda_tell(s) == refshim.MZ_TELL_ERROR and lib.mz_stream_cuda_seek(s, 0, 0) == refshim.MZ_SEEK_ERROR
    assert lib.mz_stream_cuda_is_open(s) == refshim.MZ_OPEN_ERROR
    ps = C.c_void_p(s)
    lib.mz_stream_cuda_delete(C.byref(ps))
    assert ps.value is None
    lib.mz_stream_cuda_delete(None)


def test_stream_written_by_us_read_by_reference(cu):
    """The acceptance test of the north star: the reference's inflate (zlib's, under mz_strm_zlib.c) decodes our streams
    bit-exactly, and our CRC symbol returns the reference's CRCs (pinned in tests/golden/reference_outputs.json)."""
    p, lib, tl = cu
    pinned = {e["seed"]: e["crc32"] for e in refshim.reference_outputs()["parity_crc"]}
    for wb in (-15, 31):
        for level in (1, 6):
            data = datagen.mixed(700000, wb + level + 50)
            comp, info = tl.compress(lib.mz_stream_cuda_create, data, level=level, window_bits=wb)
            out, consumed, at_end = refshim.zlib_read(comp, wb)
            assert at_end and out == data
            assert consumed == len(comp) and len(out) == len(data)
            assert pinned[wb + level + 50] == lib.mz_crypt_crc32_update(0, C.create_string_buffer(data, len(data)), len(data))


# ---- the vtbl stream: read path -------------------------------------------------------------------------------------
def test_stream_read_golden_reference_streams(cu, golden):
    p, lib, tl = cu
    for v in golden["refrun"]:
        comp = bytes.fromhex(v["stream_hex"])
        out, info = tl.decompress(lib.mz_stream_cuda_create, comp, v["size"], window_bits=v["window_bits"])
        assert info["read"] == v["size"], (v["input"], v["level"], v["window_bits"], info)
        assert zlib.crc32(out) == v["crc32"]
        assert info["total_in"] == len(comp) and info["total_out"] == v["size"] and info["close"] == 0
        assert info["read_again"] == 0  # stays at end of stream


def test_stream_read_foreign_corpus_entries(cu, golden):
    """Third-party DEFLATE entries of the reference's seed corpus: sizes and CRCs from the zip headers."""
    p, lib, tl = cu
    n = 0
    for ent in golden["foreign"]:
        if ent["method"] != 8:
            continue
        comp = bytes.fromhex(ent["payload_hex"])
        out, info = tl.decompress(lib.mz_stream_cuda_create, comp + b"PK\x01\x02 trailing central directory bytes", ent["size"])
        assert info["read"] == ent["size"] and zlib.crc32(out) == ent["crc32"], ent["name"]
        assert info["total_in"] == len(comp)  # over-read from base, exact consumed count (mz_zip.c:2100-2112)
        n += 1
    assert n >= 10


@pytest.mark.parametrize("read_size", [1, 4096, 65535])
def test_stream_read_sizes_and_windows(cu, read_size, monkeypatch):
    p, lib, tl = cu
    monkeypatch.setenv("MZ_CUDA_BATCH_KB", "256")  # force input refills and output window slides
    n = 200000 if read_size == 1 else 3000000
    data = datagen.mixed(n, 77)
    for level, wb in ((1, -15), (6, 31), (9, 15), (0, -15)):
        comp = zlib.compressobj(level, zlib.DEFLATED, wb)
        comp = comp.compress(data) + comp.flush()
        out, info = tl.decompress(lib.mz_stream_cuda_create, comp, n, window_bits=wb, read_size=read_size)
        assert info["read"] == n and out == data, (level, wb, info)
        assert info["total_in"] == len(comp) and info["total_out"] == n


def test_stream_read_parallel_copy_slices(cu):
    """reads big enough for the helper threads (>= 256 KiB) whose size is NOT a multiple of the thread count while a quarter of it IS a
    multiple of 4 KiB: the slice rounding that lost the last n mod 4 bytes in round 2 (262146 = 4 * 65536 + 2, 1048579 = 4 * 262144 + 3)"""
    p, lib, tl = cu
    data = datagen.mixed(6_000_000, 91)
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    comp = co.compress(data) + co.flush()
    for read_size in (262146, 1048579, 786433):
        out, info = tl.decompress(lib.mz_stream_cuda_create, comp, len(data), window_bits=31, read_size=read_size)
        assert info["read"] == len(data) and out == data, (read_size, info)
        assert info["total_in"] == len(comp) and info["close"] == 0


def test_stream_read_errors(cu, golden):
    """Error taxonomy observed from the reference (SURVEY.md 8c): truncated -> -5, bad trailer / wrong framing -> -3, sticky, close -> -112."""
    p, lib, tl = cu
    data = datagen.text_like(500000, 4)
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    comp = co.compress(data) + co.flush()
    out, info = tl.decompress(lib.mz_stream_cuda_create, comp[:len(comp) // 2], len(data), window_bits=31)
    assert info["read"] == refshim.MZ_BUF_ERROR or (info["read"] > 0 and info["read_again"] == refshim.MZ_BUF_ERROR)
    assert info["error"] == refshim.MZ_BUF_ERROR and info["close"] == refshim.MZ_CLOSE_ERROR
    bad = bytearray(comp)
    bad[-8] ^= 0xFF
    out, info = tl.decompress(lib.mz_stream_cuda_create, bytes(bad), len(data), window_bits=31)
    assert info["error"] == refshim.MZ_DATA_ERROR and info["close"] == refshim.MZ_CLOSE_ERROR
    raw = zlib.compressobj(6, zlib.DEFLATED, -15)
    raw = raw.compress(data) + raw.flush()
    out, info = tl.decompress(lib.mz_stream_cuda_create, raw, len(data), window_bits=31)
    assert info["read"] == refshim.MZ_DATA_ERROR
    garbage = bytes([0x07]) + b"\xff" * 100  # reserved block type 3
    out, info = tl.decompress(lib.mz_stream_cuda_create, garbage, 1000, window_bits=-15)
    assert info["error"] == refshim.MZ_DATA_ERROR
    two = comp + comp  # two gzip members: only the first is decoded (SURVEY 8c)
    out, info = tl.decompress(lib.mz_stream_cuda_create, two, len(data) * 2, window_bits=31)
    assert info["read"] == len(data) and info["total_in"] == len(comp)


def test_stream_read_total_in_max(cu):
    p, lib, tl = cu
    data = datagen.text_like(100000, 8)
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    out, info = tl.decompress(lib.mz_stream_cuda_create, comp + b"\x00" * 1000, len(data), total_in_max=len(comp))
    assert info["read"] == len(data) and out == data and info["base_tell"] == len(comp)


def test_full_roundtrip_both_ways_on_gpu(cu):
    """write (GPU deflate) -> read (GPU inflate), gzip, through the vtbl both ways; checksum of the result."""
    p, lib, tl = cu
    data = datagen.mixed(5 << 20, 123)
    comp, info = tl.compress(lib.mz_stream_cuda_create, data, level=1, window_bits=31, write_size=1 << 20)
    out, rinfo = tl.decompress(lib.mz_stream_cuda_create, comp, len(data), window_bits=31, read_size=65535)
    assert rinfo["read"] == len(data) and out == data and rinfo["total_in"] == len(comp)


def test_device_inflate_batch_of_streams(cu, torch_cuda, orc):
    """K5 on many independent streams at once (zip-extract shape)."""
    p, lib, _ = cu
    torch = torch_cuda
    blobs = [datagen.mixed(20000 + 997 * i, 300 + i) for i in range(40)]
    comps = []
    for i, b in enumerate(blobs):
        co = zlib.compressobj(1 + (i % 9), zlib.DEFLATED, -15)
        comps.append(co.compress(b) + co.flush())
    in_off, pos = [], 0
    for c in comps:
        in_off.append(pos)
        pos += (len(c) + 64 + 15) // 16 * 16
    cin = bytearray(pos + 64)
    for o, c in zip(in_off, comps):
        cin[o:o + len(c)] = c
    out_off, opos = [], 0
    for b in blobs:
        out_off.append(opos)
        opos += len(b) + 512
    d_in = _dev(torch, bytes(cin))
    d_out = torch.zeros(opos, dtype=torch.uint8, device="cuda")
    jobs = (p.InflateJob * len(blobs))()
    for i in range(len(blobs)):
        jobs[i] = p.InflateJob(d_in.data_ptr() + in_off[i], 0, len(comps[i]), d_out.data_ptr() + out_off[i], 0, len(blobs[i]), 1, 0)
    d_jobs = _dev(torch, bytes(jobs))
    d_states = torch.zeros(C.sizeof(p.InflateState) * len(blobs), dtype=torch.uint8, device="cuda")
    p.check(lib.mz_cuda_inflate_streams(d_jobs.data_ptr(), d_states.data_ptr(), len(blobs), None))
    torch.cuda.synchronize()
    raw = d_states.cpu().numpy().tobytes()
    outs = d_out.cpu().numpy()
    for i, b in enumerate(blobs):
        st = p.InflateState.from_buffer_copy(raw[i * C.sizeof(p.InflateState):(i + 1) * C.sizeof(p.InflateState)])
        assert st.status == 1 and st.out_pos == len(b) and (st.in_bitpos + 7) // 8 == len(comps[i]), i
        assert outs[out_off[i]:out_off[i] + len(b)].tobytes() == b
