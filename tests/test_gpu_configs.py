"""GPU tests shaped like BASELINE.json's five configurations (sizes reduced where the full size would take minutes;
the checks are size-independent: round trips through the REFERENCE codec, CRC of the whole == fold of the chunk CRCs).
"""
import ctypes as C
import zlib

import pytest

import datagen
import textgen
import refshim

pytestmark = pytest.mark.gpu

MiB = 1 << 20


@pytest.fixture(scope="module")
def env(built):
    import torch
    import cuharness
    p = cuharness.pkg()
    lib = p.load()
    assert lib.mz_cuda_init() == 0
    torch.cuda.set_device(0)
    return p, lib, cuharness.TestLib(), torch


def _host_bytes(t):
    return bytes(t.cpu().numpy().tobytes())


def test_c1_crc32_64mib_through_the_replaced_symbol(env, orc):
    """configs[0]: CRC32 of a 64 MiB buffer via mz_crypt_crc32_update (one call, host pointer)."""
    p, lib, tl, torch = env
    n = 64 * MiB
    src = textgen.device(n, seed=5)
    torch.cuda.synchronize()
    host = _host_bytes(src)
    buf = C.create_string_buffer(host, n)
    got = lib.mz_crypt_crc32_update(0, buf, n)
    assert got == zlib.crc32(host) == orc.crc32(0, host)
    assert p.crc32_device(src, n) == got
    zeros = torch.zeros(n, dtype=torch.uint8, device="cuda")  # value independence
    assert p.crc32_device(zeros, n) == zlib.crc32(bytes(n))


def test_c2_minigzip_level6_text_through_vtbl(env):
    """configs[1] shape: gzip (window_bits 31) level 6 of synthetic text, 16 KiB writes like mz_stream_copy_stream_to_end;
    the reference's reader (zlib's inflate) must reproduce the input (size 64 MiB here instead of 256 MiB)."""
    p, lib, tl, torch = env
    n = 64 * MiB
    host = _host_bytes(textgen.device(n, seed=6))
    comp, info = tl.compress(lib.mz_stream_cuda_create, host, level=6, window_bits=31, write_size=16384)
    assert info["total_in"] == n and info["total_out"] == len(comp) and info["close"] == 0
    assert comp[:4] == b"\x1f\x8b\x08\x00" and int.from_bytes(comp[-4:], "little") == n
    assert int.from_bytes(comp[-8:-4], "little") == zlib.crc32(host)
    out, consumed, at_end = refshim.zlib_read(comp, 31)
    assert at_end and len(out) == n and zlib.crc32(out) == zlib.crc32(host)
    assert consumed == len(comp)
    assert len(comp) < 0.55 * n


def test_c3_inflate_reference_gz_through_vtbl(env):
    """configs[2] shape: one multi-block gzip member written by the REFERENCE (level 6, no sync points) decoded by
    mz_stream_cuda_read in 16 KiB reads (128 MiB here instead of 4 GiB; ISIZE-mod-2^32 is covered by the trailer logic).
    The member is rebuilt with zlib and proven to be the reference's by its pinned digest."""
    p, lib, tl, torch = env
    pinned = refshim.reference_outputs()["c3_member"]
    n = 128 * MiB
    assert (pinned["n"], pinned["text_seed"], pinned["level"], pinned["window_bits"]) == (n, 7, 6, 31)
    host = _host_bytes(textgen.device(n, seed=7))
    assert zlib.crc32(host) == pinned["crc32"]
    comp = refshim.zlib_stream(host, 6, 31)
    assert refshim.is_reference_stream(comp, pinned)
    out, info = tl.decompress(lib.mz_stream_cuda_create, comp, n, window_bits=31, read_size=16384)
    assert info["read"] == n and info["total_in"] == len(comp) and info["total_out"] == n and info["close"] == 0
    assert zlib.crc32(out) == zlib.crc32(host)


def test_c4_zip_entries_batch(env, orc):
    """configs[3] shape: many independent 64 KiB entries, raw deflate level 6 + CRC each, one launch (4000 entries here)."""
    p, lib, tl, torch = env
    n_ent, ent = 4000, 65536
    total = n_ent * ent
    src = torch.empty(total, dtype=torch.uint8, device="cuda")
    textgen.device_into(src.data_ptr(), total * 7 // 10, 11)
    src[total * 7 // 10:] = torch.randint(0, 256, (total - total * 7 // 10,), dtype=torch.uint8, device="cuda")  # incompressible tail
    d_off = torch.arange(n_ent, dtype=torch.int64, device="cuda") * ent
    d_len = torch.full((n_ent,), ent, dtype=torch.int32, device="cuda")
    d_flags = torch.ones(n_ent, dtype=torch.uint8, device="cuda")
    stride = int(lib.mz_cuda_deflate_slot_bound(ent))
    slots = torch.empty(n_ent * stride, dtype=torch.uint8, device="cuda")
    out_len = torch.empty(n_ent, dtype=torch.int32, device="cuda")
    res = torch.empty(n_ent, dtype=torch.int32, device="cuda")
    crc = torch.empty(n_ent, dtype=torch.int32, device="cuda")
    p.check(lib.mz_cuda_deflate_chunks(src.data_ptr(), 0, 0, d_off.data_ptr(), d_len.data_ptr(), d_flags.data_ptr(), n_ent, 0, 6,
                                       slots.data_ptr(), stride, out_len.data_ptr(), None))
    p.check(lib.mz_cuda_crc32_segments(src.data_ptr(), 0, 0, d_off.data_ptr(), d_len.data_ptr(), n_ent, res.data_ptr(), crc.data_ptr(), None))
    torch.cuda.synchronize()
    host = src.cpu().numpy()
    lens = out_len.cpu().numpy()
    crcs = crc.cpu().numpy()
    raw = slots.cpu().numpy()
    assert int(lens.max()) <= stride and int(lens[:n_ent // 2].mean()) < ent * 0.6
    for i in list(range(0, n_ent, 97)) + [n_ent - 1]:
        blob = host[i * ent:(i + 1) * ent].tobytes()
        comp = raw[i * stride:i * stride + int(lens[i])].tobytes()
        assert zlib.decompress(comp, -15) == blob, i
        assert (int(crcs[i]) & 0xFFFFFFFF) == zlib.crc32(blob)
    # every entry decodes on the GPU as well (K5 batch), compared by CRC
    jobs = (p.InflateJob * n_ent)()
    d_out = torch.zeros(n_ent * (ent + 512), dtype=torch.uint8, device="cuda")
    padded = torch.zeros(n_ent * stride + 64, dtype=torch.uint8, device="cuda")
    padded[:n_ent * stride] = slots
    for i in range(n_ent):
        jobs[i] = p.InflateJob(padded.data_ptr() + i * stride, 0, int(lens[i]), d_out.data_ptr() + i * (ent + 512), 0, ent, 1, 0)
    import numpy as np
    d_jobs = torch.from_numpy(np.frombuffer(bytes(jobs), dtype=np.uint8).copy()).cuda()
    d_states = torch.zeros(C.sizeof(p.InflateState) * n_ent, dtype=torch.uint8, device="cuda")
    p.check(lib.mz_cuda_inflate_streams(d_jobs.data_ptr(), d_states.data_ptr(), n_ent, None))
    torch.cuda.synchronize()
    o_off = torch.arange(n_ent, dtype=torch.int64, device="cuda") * (ent + 512)
    crc2 = torch.empty(n_ent, dtype=torch.int32, device="cuda")
    p.check(lib.mz_cuda_crc32_segments(d_out.data_ptr(), 0, 0, o_off.data_ptr(), d_len.data_ptr(), n_ent, res.data_ptr(), crc2.data_ptr(), None))
    torch.cuda.synchronize()
    assert torch.equal(crc, crc2)


def test_c5_chunked_level1_with_crc_fold(env):
    """configs[4] shape: one long buffer, independent 64 KiB chunks, level 1 + CRC per chunk + fold + join, in two
    batches (non-final then final) like two GPUs' shards; the reference reader decodes the concatenation (512 MiB)."""
    p, lib, tl, torch = env
    n = 512 * MiB
    half = n // 2
    src = textgen.device(n, seed=8)
    torch.cuda.synchronize()
    b = p.DeflateBatch(half)
    parts, crcs = [], []
    for i, off in enumerate((0, half)):
        k = b.compress(src[off:off + half], half, level=1, final=(i == 1))
        joined, crc = b.result(k)
        parts.append(_host_bytes(joined))
        crcs.append(crc)
    comp = b"".join(parts)
    host = _host_bytes(src)
    whole = zlib.crc32(host)
    assert lib.mz_cuda_crc32_combine(crcs[0], crcs[1], half) == whole  # checksum of checksums
    d = zlib.decompressobj(-15)
    crc, total = 0, 0
    for o in range(0, len(comp), 8 * MiB):
        piece = d.decompress(comp[o:o + 8 * MiB])
        crc = zlib.crc32(piece, crc)
        total += len(piece)
    piece = d.flush()
    crc = zlib.crc32(piece, crc)
    total += len(piece)
    assert d.eof and total == n and crc == whole
    # and the second batch on its own, as the reference's stream reader (zlib's inflate) would take it
    out, _, at_end = refshim.zlib_read(parts[1], -15)
    assert at_end and zlib.crc32(out) == zlib.crc32(host[half:])


def test_c3_long_member_speculative_rounds_match_serial(env, monkeypatch):
    """the segment-speculative rounds (K6) and the serial decoder must deliver identical bytes and totals for the same
    foreign member; zlib level 1/6/9 members, Z_FULL_FLUSH-riddled members and a member with a long stored run inside"""
    p, lib, tl, torch = env
    n = 48 * MiB
    text = _host_bytes(textgen.device(n, seed=17))
    noise = datagen.random_bytes(6 * MiB, seed=5)
    cases = []
    for level in (1, 6, 9):
        co = zlib.compressobj(level, zlib.DEFLATED, 31)
        cases.append((text, co.compress(text) + co.flush()))
    for level, nbytes in ((6, 12 * MiB), (9, 3 * MiB), (1, 700_000)):  # medium members: K6 on the small windows (zip-entry sizes)
        co = zlib.compressobj(level, zlib.DEFLATED, 31)
        cases.append((text[:nbytes], co.compress(text[:nbytes]) + co.flush()))
    mixed = text[:20 * MiB] + noise + text[20 * MiB:30 * MiB]  # stored blocks in the middle: the rounds must hand over and resume
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    cases.append((mixed, co.compress(mixed) + co.flush()))
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    parts = []
    for o in range(0, 24 * MiB, 300_000):
        parts.append(co.compress(text[o:o + 300_000]))
        parts.append(co.flush(zlib.Z_FULL_FLUSH))
    parts.append(co.flush())
    cases.append((text[:(24 * MiB + 299_999) // 300_000 * 300_000][:24 * MiB + 300_000], b"".join(parts)))
    for plain, comp in cases:
        plain = zlib.decompress(comp, 31)  # ground truth straight from zlib
        outs = []
        for spec in ("1", "0"):
            monkeypatch.setenv("MZ_CUDA_SPEC", spec)
            out, info = tl.decompress(lib.mz_stream_cuda_create, comp, len(plain), window_bits=31, read_size=1 << 20)
            assert info["read"] == len(plain) and info["total_in"] == len(comp) and info["total_out"] == len(plain) and info["close"] == 0, (spec, info)
            outs.append(zlib.crc32(out))
        assert outs[0] == outs[1] == zlib.crc32(plain)
    # a corrupted long member: same error class either way, and no wrong bytes before it
    plain, comp = cases[1]
    bad = bytearray(comp)
    for k in range(len(bad) // 2, len(bad) // 2 + 64):
        bad[k] ^= 0xA5
    res = []
    for spec in ("1", "0"):
        monkeypatch.setenv("MZ_CUDA_SPEC", spec)
        out, info = tl.decompress(lib.mz_stream_cuda_create, bytes(bad), len(plain), window_bits=31, read_size=1 << 20)
        res.append((info["read"], info["error"]))
        good = out if out else b""
        assert plain.startswith(good)
    assert res[0][1] != 0 and res[1][1] != 0


def test_c3_abandoned_long_read_leaves_the_workspace_usable(env):
    """a caller may stop reading in the middle of a long member (a speculative round is then still in flight): close must
    return cleanly and the pooled workspace must serve the next streams -- a long one, then a tiny one -- correctly"""
    p, lib, tl, torch = env
    import cuharness
    text = _host_bytes(textgen.device(40 * MiB, seed=23))
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    comp = co.compress(text) + co.flush()
    src, keep = tl.source(comp)
    s = lib.mz_stream_cuda_create()
    assert tl.lib.mzt_set_prop(s, p.MZ_STREAM_PROP_COMPRESS_WINDOW, 31) == 0
    tl.lib.mzt_set_base(s, src)
    assert tl.lib.mzt_open(s, None, p.MZ_OPEN_MODE_READ) == 0
    buf = C.create_string_buffer(1 << 20)
    got = tl.lib.mzt_read(s, buf, 1 << 20)
    assert got > 0 and text.startswith(buf.raw[:got])
    assert tl.lib.mzt_close(s) == 0  # 39 MiB never read
    tl.delete(s)
    tl.delete(src)
    out, info = tl.decompress(lib.mz_stream_cuda_create, comp, len(text), window_bits=31, read_size=300_000)
    assert info["read"] == len(text) and zlib.crc32(out) == zlib.crc32(text) and info["total_in"] == len(comp)
    small = zlib.compress(b"tiny stream after a big one " * 40, 9)
    out, info = tl.decompress(lib.mz_stream_cuda_create, small, 2000, window_bits=15, read_size=100)
    assert out == b"tiny stream after a big one " * 40 and info["total_in"] == len(small) and info["close"] == 0
