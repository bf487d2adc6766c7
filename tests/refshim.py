"""ctypes access to the CHECKERS (test infrastructure only):

RefLib    : oracle/_ref/libmzref.so -- the reference's own mz_strm_zlib.c / mz_crypt.c / mz_strm*.c
            compiled from /root/reference + system zlib 1.3 (oracle/Makefile).
OracleLib : oracle/liboracle.so -- the C restatement (oracle/mzoracle.c).

The generic mz_stream_* dispatchers of RefLib (mz_strm.c:20-130) work on ANY object whose first
member is an mz_stream {vtbl, base}, so the same calls drive the reference codec and mz_strm_cuda.
"""
import ctypes as C
import hashlib
import json
import os
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MZ_OK = 0
MZ_STREAM_ERROR, MZ_DATA_ERROR, MZ_MEM_ERROR, MZ_BUF_ERROR = -1, -3, -4, -5
MZ_PARAM_ERROR, MZ_EXIST_ERROR, MZ_SUPPORT_ERROR = -102, -107, -109
MZ_OPEN_ERROR, MZ_CLOSE_ERROR, MZ_SEEK_ERROR, MZ_TELL_ERROR, MZ_WRITE_ERROR = -111, -112, -113, -114, -116
MZ_OPEN_MODE_READ, MZ_OPEN_MODE_WRITE, MZ_OPEN_MODE_CREATE = 0x01, 0x02, 0x08
MZ_SEEK_SET = 0
PROP_TOTAL_IN, PROP_TOTAL_IN_MAX, PROP_TOTAL_OUT, PROP_TOTAL_OUT_MAX, PROP_HEADER_SIZE = 1, 2, 3, 4, 5
PROP_COMPRESS_LEVEL, PROP_COMPRESS_METHOD, PROP_COMPRESS_WINDOW = 9, 10, 11


def ref_available():
    return os.path.exists(os.path.join(ROOT, "oracle/_ref/libmzref.so"))


# -- the reference's outputs without a reference build ---------------------------------------------------------------
# mz_strm_zlib.c is a framing layer over zlib's deflate (memLevel 8, default strategy) and inflate, the same calls
# CPython's zlib makes. tests/golden/reference_outputs.json pins what the reference returned for the tests' seeded inputs
# (tests/golden/make_golden.py); a stream rebuilt here is the reference's when its length and SHA-256 match.
def reference_outputs():
    return json.load(open(os.path.join(ROOT, "tests/golden/reference_outputs.json")))


def zlib_stream(data, level, window_bits):
    co = zlib.compressobj(level, zlib.DEFLATED, window_bits)
    return co.compress(data) + co.flush()


def is_reference_stream(stream, pinned):
    return len(stream) == pinned["size"] and hashlib.sha256(stream).hexdigest() == pinned["sha256"]


def zlib_read(comp, window_bits):
    """The reference reader's decode of one stream: (bytes, compressed bytes consumed, end of stream reached)."""
    d = zlib.decompressobj(window_bits)
    out = d.decompress(comp) + d.flush()
    return out, len(comp) - len(d.unused_data), d.eof


def _sig(fn, res, args):
    fn.restype = res
    fn.argtypes = args
    return fn


class RefLib:
    def __init__(self, path=None):
        path = path or os.path.join(ROOT, "oracle/_ref/libmzref.so")
        self.lib = L = C.CDLL(path, mode=os.RTLD_LOCAL if hasattr(os, "RTLD_LOCAL") else 0)
        vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
        for name in ("mz_stream_mem_create", "mz_stream_zlib_create", "mz_stream_raw_create"):
            _sig(getattr(L, name), vp, [])
        _sig(L.mz_stream_open, i32, [vp, C.c_char_p, i32])
        _sig(L.mz_stream_is_open, i32, [vp])
        _sig(L.mz_stream_read, i32, [vp, vp, i32])
        _sig(L.mz_stream_write, i32, [vp, vp, i32])
        _sig(L.mz_stream_tell, i64, [vp])
        _sig(L.mz_stream_seek, i32, [vp, i64, i32])
        _sig(L.mz_stream_close, i32, [vp])
        _sig(L.mz_stream_error, i32, [vp])
        _sig(L.mz_stream_set_base, i32, [vp, vp])
        _sig(L.mz_stream_get_prop_int64, i32, [vp, i32, C.POINTER(i64)])
        _sig(L.mz_stream_set_prop_int64, i32, [vp, i32, i64])
        _sig(L.mz_stream_delete, None, [C.POINTER(vp)])
        _sig(L.mz_stream_copy_stream_to_end, i32, [vp, vp, vp, vp])
        _sig(L.mz_stream_mem_set_buffer, None, [vp, vp, i32])
        _sig(L.mz_stream_mem_get_buffer, i32, [vp, C.POINTER(vp)])
        _sig(L.mz_stream_mem_get_buffer_length, None, [vp, C.POINTER(i32)])
        _sig(L.mz_stream_mem_set_grow_size, None, [vp, i32])
        _sig(L.mz_crypt_crc32_update, C.c_uint32, [C.c_uint32, vp, i32])

    # -- generic helpers over any stream object --------------------------------------------
    def get_prop(self, strm, prop):
        v = C.c_int64(-999)
        err = self.lib.mz_stream_get_prop_int64(strm, prop, C.byref(v))
        return err, v.value

    def delete(self, strm):
        p = C.c_void_p(strm)
        self.lib.mz_stream_delete(C.byref(p))
        return p.value

    def mem_from_bytes(self, data):
        m = self.lib.mz_stream_mem_create()
        keep = C.create_string_buffer(data, len(data)) if len(data) else C.create_string_buffer(1)
        self.lib.mz_stream_mem_set_buffer(m, keep, len(data))
        assert self.lib.mz_stream_open(m, None, MZ_OPEN_MODE_READ) == MZ_OK
        return m, keep

    def mem_sink(self, grow=1 << 20):
        m = self.lib.mz_stream_mem_create()
        self.lib.mz_stream_mem_set_grow_size(m, grow)
        assert self.lib.mz_stream_open(m, None, MZ_OPEN_MODE_CREATE) == MZ_OK
        return m

    def mem_bytes(self, m):
        ln = C.c_int32(0)
        self.lib.mz_stream_mem_get_buffer_length(m, C.byref(ln))
        p = C.c_void_p()
        self.lib.mz_stream_mem_get_buffer(m, C.byref(p))
        return C.string_at(p, ln.value) if ln.value else b""

    def write_all(self, strm, data, write_size):
        buf = C.create_string_buffer(data, len(data)) if len(data) else C.create_string_buffer(1)
        base = C.addressof(buf)
        pos = 0
        while pos < len(data):
            n = min(write_size, len(data) - pos)
            r = self.lib.mz_stream_write(strm, base + pos, n)
            if r != n:
                return r
            pos += n
        return len(data)

    def read_all(self, strm, read_size=16384, limit=None):
        out = bytearray()
        buf = C.create_string_buffer(read_size)
        while True:
            r = self.lib.mz_stream_read(strm, buf, read_size)
            if r < 0:
                return r, bytes(out)
            if r == 0:
                return 0, bytes(out)
            out += buf.raw[:r]
            if limit is not None and len(out) > limit:
                return -999, bytes(out)

    # -- the reference path --------------------------------------------------------------------
    def compress_with(self, create_fn, data, level=6, window_bits=-15, write_size=16384):
        """create -> set_prop -> set_base(mem) -> open(WRITE) -> write* -> close (test_stream_compress.cc:64-76)."""
        sink = self.mem_sink()
        s = create_fn()
        assert s
        assert self.lib.mz_stream_set_prop_int64(s, PROP_COMPRESS_LEVEL, level) == MZ_OK
        assert self.lib.mz_stream_set_prop_int64(s, PROP_COMPRESS_WINDOW, window_bits) == MZ_OK
        self.lib.mz_stream_set_base(s, sink)
        err = self.lib.mz_stream_open(s, None, MZ_OPEN_MODE_WRITE)
        assert err == MZ_OK, err
        assert self.write_all(s, data, write_size) == len(data)
        cerr = self.lib.mz_stream_close(s)
        tin = self.get_prop(s, PROP_TOTAL_IN)
        tout = self.get_prop(s, PROP_TOTAL_OUT)
        out = self.mem_bytes(sink)
        info = {"close": cerr, "total_in": tin[1], "total_out": tout[1], "sink_tell": self.lib.mz_stream_tell(sink)}
        self.delete(s)
        self.lib.mz_stream_close(sink)
        self.delete(sink)
        return out, info

    def decompress_with(self, create_fn, comp, window_bits=-15, read_size=16384):
        src, keep = self.mem_from_bytes(comp)
        s = create_fn()
        assert self.lib.mz_stream_set_prop_int64(s, PROP_COMPRESS_WINDOW, window_bits) == MZ_OK
        self.lib.mz_stream_set_base(s, src)
        assert self.lib.mz_stream_open(s, None, MZ_OPEN_MODE_READ) == MZ_OK
        err, out = self.read_all(s, read_size)
        cerr = self.lib.mz_stream_close(s)
        info = {"read_err": err, "close": cerr, "total_in": self.get_prop(s, PROP_TOTAL_IN)[1],
                "total_out": self.get_prop(s, PROP_TOTAL_OUT)[1], "error": self.lib.mz_stream_error(s),
                "base_tell": self.lib.mz_stream_tell(src)}
        self.delete(s)
        self.lib.mz_stream_close(src)
        self.delete(src)
        return out, info

    def zlib_compress(self, data, level=6, window_bits=-15, write_size=16384):
        return self.compress_with(self.lib.mz_stream_zlib_create, data, level, window_bits, write_size)[0]

    def zlib_decompress(self, comp, window_bits=-15, read_size=16384):
        out, info = self.decompress_with(self.lib.mz_stream_zlib_create, comp, window_bits, read_size)
        if info["read_err"] != 0:
            raise ValueError("reference inflate failed: %d" % info["read_err"])
        return out

    def crc32(self, value, data):
        buf = C.create_string_buffer(data, len(data)) if len(data) else C.create_string_buffer(1)
        return self.lib.mz_crypt_crc32_update(value, buf, len(data))


class OracleLib:
    WRAP_RAW, WRAP_ZLIB, WRAP_GZIP = 0, 1, 2

    def __init__(self, path=None):
        path = path or os.path.join(ROOT, "oracle/liboracle.so")
        self.lib = L = C.CDLL(path)
        vp, sz = C.c_void_p, C.c_size_t
        _sig(L.orc_crc32_update, C.c_uint32, [C.c_uint32, vp, sz])
        _sig(L.orc_crc32_combine, C.c_uint32, [C.c_uint32, C.c_uint32, C.c_uint64])
        _sig(L.orc_inflate, C.c_int, [vp, sz, vp, sz, C.c_int, C.POINTER(sz), C.POINTER(sz)])
        _sig(L.orc_deflate, C.c_int64, [vp, sz, vp, sz, C.c_int, C.c_int])
        _sig(L.orc_deflate_bound, sz, [sz])
        _sig(L.orc_inflate_blocks, C.c_int64, [vp, sz, C.c_int, vp, sz, C.POINTER(sz)])

    @staticmethod
    def wrap_of(window_bits):
        return 0 if window_bits < 0 else (2 if window_bits > 15 else 1)

    def crc32(self, value, data):
        data = bytes(data)
        return self.lib.orc_crc32_update(value, data, len(data))

    def crc32_combine(self, a, b, len_b):
        return self.lib.orc_crc32_combine(a, b, len_b)

    def inflate(self, comp, out_cap, window_bits=-15):
        """returns (err, out_bytes, consumed)"""
        comp = bytes(comp)
        out = C.create_string_buffer(max(out_cap, 1))
        cons, prod = C.c_size_t(0), C.c_size_t(0)
        err = self.lib.orc_inflate(comp, len(comp), out, out_cap, self.wrap_of(window_bits), C.byref(cons), C.byref(prod))
        return err, out.raw[:prod.value], cons.value

    def deflate(self, data, level=6, window_bits=-15):
        data = bytes(data)
        cap = self.lib.orc_deflate_bound(len(data))
        out = C.create_string_buffer(cap)
        n = self.lib.orc_deflate(data, len(data), out, cap, level, self.wrap_of(window_bits))
        if n < 0:
            raise ValueError("orc_deflate %d" % n)
        return out.raw[:n]

    def blocks(self, comp, window_bits=-15, max_blocks=1 << 16):
        class BI(C.Structure):
            _fields_ = [("start_bit", C.c_uint64), ("out_bytes", C.c_uint64), ("type", C.c_int32), ("final", C.c_int32)]
        arr = (BI * max_blocks)()
        prod = C.c_size_t(0)
        comp = bytes(comp)
        n = self.lib.orc_inflate_blocks(comp, len(comp), self.wrap_of(window_bits), arr, max_blocks, C.byref(prod))
        if n < 0:
            raise ValueError("orc_inflate_blocks %d" % n)
        return [(arr[i].start_bit, arr[i].out_bytes, arr[i].type, arr[i].final) for i in range(min(n, max_blocks))], prod.value
