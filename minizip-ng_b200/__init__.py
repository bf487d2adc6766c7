"""minizip-ng_b200 -- host-side Python mirror of the B200 DEFLATE + CRC-32 backend.

The product is the C-ABI shared library ``libmz_strm_cuda.so`` (include/mz_strm_cuda.h,
include/mz_cuda_batch.h).  This package only (a) loads it with ctypes, (b) wraps device buffers in
torch tensors for the bench / multi-GPU plumbing, (c) mirrors the reference's stream interface names so
tests read like test/test_stream_compress.cc.  There is no Python or CPU codec here: if the library is
missing or no sm_100 GPU is usable, calls raise.

Import note: the directory name contains a hyphen (the project name); load it with
``importlib`` (see __graft_entry__._load_pkg) -- it registers itself as ``minizip_ng_b200``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmz_strm_cuda.so")

MZ_OK = 0
MZ_DATA_ERROR, MZ_MEM_ERROR, MZ_BUF_ERROR = -3, -4, -5
MZ_SUPPORT_ERROR, MZ_OPEN_ERROR, MZ_CLOSE_ERROR = -109, -111, -112
MZ_OPEN_MODE_READ, MZ_OPEN_MODE_WRITE = 0x01, 0x02
MZ_STREAM_PROP_TOTAL_IN, MZ_STREAM_PROP_TOTAL_IN_MAX, MZ_STREAM_PROP_TOTAL_OUT = 1, 2, 3
MZ_STREAM_PROP_COMPRESS_LEVEL, MZ_STREAM_PROP_COMPRESS_WINDOW = 9, 11
CHUNK_MAX = 65536
FLAG_FINAL = 1
FLAG_DICT = 2  # the buffer is ONE stream: at levels 6-9 a chunk may refer back into the 32 KiB before it

_lib = None


class InflateJob(C.Structure):
    _fields_ = [("d_in", C.c_void_p), ("in_base", C.c_uint64), ("in_avail", C.c_uint64), ("d_out", C.c_void_p),
                ("out_base", C.c_uint64), ("out_cap", C.c_uint64), ("in_final", C.c_uint32), ("flags", C.c_uint32)]


class InflateState(C.Structure):
    _fields_ = [("in_bitpos", C.c_uint64), ("out_pos", C.c_uint64), ("status", C.c_int32), ("why", C.c_int32),
                ("phase", C.c_uint32), ("last_block", C.c_uint32), ("stored_remaining", C.c_uint32), ("nlit", C.c_uint32),
                ("ndist", C.c_uint32), ("blocks", C.c_uint32), ("lens", C.c_uint8 * 320)]


EXPORTS = [
    # include/mz_strm_cuda.h
    "mz_stream_cuda_open", "mz_stream_cuda_is_open", "mz_stream_cuda_read", "mz_stream_cuda_write", "mz_stream_cuda_tell",
    "mz_stream_cuda_seek", "mz_stream_cuda_close", "mz_stream_cuda_error", "mz_stream_cuda_get_prop_int64",
    "mz_stream_cuda_set_prop_int64", "mz_stream_cuda_create", "mz_stream_cuda_delete", "mz_stream_cuda_get_interface",
    "mz_crypt_crc32_update",
    # include/mz_cuda_batch.h
    "mz_cuda_init", "mz_cuda_device_count", "mz_cuda_set_device", "mz_cuda_get_device", "mz_cuda_last_error", "mz_cuda_sm_count", "mz_cuda_malloc",
    "mz_cuda_free", "mz_cuda_host_alloc", "mz_cuda_host_free", "mz_cuda_memcpy_h2d", "mz_cuda_memcpy_d2h", "mz_cuda_memcpy_d2d",
    "mz_cuda_memset", "mz_cuda_host_is_pinned", "mz_cuda_stream_sync", "mz_cuda_stream_create", "mz_cuda_stream_destroy",
    "mz_cuda_event_create", "mz_cuda_event_destroy", "mz_cuda_event_record", "mz_cuda_event_sync", "mz_cuda_event_query", "mz_cuda_event_elapsed_ms",
    "mz_cuda_crc32_segments", "mz_cuda_crc32_fold", "mz_cuda_crc32_device", "mz_cuda_crc32_device_stream", "mz_cuda_crc32_combine",
    "mz_cuda_deflate_slot_bound", "mz_cuda_deflate_chunks", "mz_cuda_concat", "mz_cuda_inflate_streams",
    "mz_cuda_inflate_spec_workspace_bytes", "mz_cuda_inflate_spec_round", "mz_cuda_sha256_batch",
    "mz_cuda_wzaes_derive", "mz_cuda_wzaes_ctr", "mz_cuda_wzaes_hmac",
    "mz_cuda_pkcrypt_workspace_bytes", "mz_cuda_pkcrypt_encrypt", "mz_cuda_pkcrypt_decrypt",
    "mz_cuda_gather_region_bound", "mz_cuda_deflate_sharded", "mz_cuda_ipc_export", "mz_cuda_ipc_open", "mz_cuda_ipc_close", "mz_cuda_memcpy_peer",
    "mz_cuda_stream_wait_event", "mz_cuda_gather", "mz_cuda_scatter_blobs",
    # include/mz_zip_cuda.h
    "mz_zip_cuda_add_buffers", "mz_zip_cuda_add_buffers_ex", "mz_zip_cuda_write_archive", "mz_zip_cuda_trim", "mz_zip_cuda_write_archive_aes", "mz_zip_cuda_extract_all",
    "mz_zip_cuda_extract_all_aes", "mz_zip_cuda_abi_file_info_size", "mz_zip_cuda_write_archive_pkcrypt", "mz_zip_cuda_extract_all_encrypted",
]


def load():
    """Load the product library; fail loudly if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libmz_strm_cuda.so is missing: run __graft_entry__.build() (nvcc, sm_100a). "
                           "There is no CPU fallback.")
    _lib = configure(C.CDLL(LIB_PATH))
    return _lib


def configure(L):
    """ctypes prototypes of the C-ABI on an already loaded library (the product .so, or -- in the CPU test suite -- the same
    sources built against the execution-model emulator, tests/emu/libmz_strm_emu.so)."""
    vp, i32, i64, u32, u64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_size_t

    def sig(name, res, args):
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args

    sig("mz_stream_cuda_open", i32, [vp, C.c_char_p, i32])
    sig("mz_stream_cuda_is_open", i32, [vp])
    sig("mz_stream_cuda_read", i32, [vp, vp, i32])
    sig("mz_stream_cuda_write", i32, [vp, vp, i32])
    sig("mz_stream_cuda_tell", i64, [vp])
    sig("mz_stream_cuda_seek", i32, [vp, i64, i32])
    sig("mz_stream_cuda_close", i32, [vp])
    sig("mz_stream_cuda_error", i32, [vp])
    sig("mz_stream_cuda_get_prop_int64", i32, [vp, i32, C.POINTER(i64)])
    sig("mz_stream_cuda_set_prop_int64", i32, [vp, i32, i64])
    sig("mz_stream_cuda_create", vp, [])
    sig("mz_stream_cuda_delete", None, [C.POINTER(vp)])
    sig("mz_stream_cuda_get_interface", vp, [])
    sig("mz_crypt_crc32_update", u32, [u32, vp, i32])
    sig("mz_cuda_init", i32, [])
    sig("mz_cuda_device_count", i32, [])
    sig("mz_cuda_set_device", i32, [i32])
    sig("mz_cuda_last_error", C.c_char_p, [])
    sig("mz_cuda_sm_count", i32, [])
    sig("mz_cuda_malloc", vp, [sz])
    sig("mz_cuda_free", None, [vp])
    sig("mz_cuda_host_alloc", vp, [sz])
    sig("mz_cuda_host_free", None, [vp])
    sig("mz_cuda_memcpy_h2d", i32, [vp, vp, sz, vp])
    sig("mz_cuda_memcpy_d2h", i32, [vp, vp, sz, vp])
    sig("mz_cuda_memcpy_d2d", i32, [vp, vp, sz, vp])
    sig("mz_cuda_memset", i32, [vp, C.c_int, sz, vp])
    sig("mz_cuda_host_is_pinned", i32, [vp])
    sig("mz_cuda_stream_sync", i32, [vp])
    sig("mz_cuda_stream_create", vp, [])
    sig("mz_cuda_stream_destroy", None, [vp])
    sig("mz_cuda_event_create", vp, [])
    sig("mz_cuda_event_destroy", None, [vp])
    sig("mz_cuda_event_record", i32, [vp, vp])
    sig("mz_cuda_event_sync", i32, [vp])
    sig("mz_cuda_event_elapsed_ms", C.c_float, [vp, vp])
    sig("mz_cuda_crc32_segments", i32, [vp, u64, u64, vp, vp, u32, vp, vp, vp])
    sig("mz_cuda_crc32_fold", i32, [vp, u32, u64, u64, vp, vp])
    sig("mz_cuda_crc32_device", i32, [vp, u64, u32, C.POINTER(u32)])
    sig("mz_cuda_crc32_combine", u32, [u32, u32, u64])
    sig("mz_cuda_deflate_slot_bound", u64, [u32])
    sig("mz_cuda_deflate_chunks", i32, [vp, u64, u32, vp, vp, vp, u32, u32, i32, vp, u64, vp, vp])
    sig("mz_cuda_concat", i32, [vp, u64, vp, u32, vp, vp, vp])
    sig("mz_cuda_inflate_streams", i32, [vp, vp, u32, vp])
    sig("mz_cuda_sha256_batch", i32, [vp, vp, vp, u32, vp, vp])
    sig("mz_cuda_wzaes_derive", i32, [vp, u32, vp, u32, u32, vp, vp])
    sig("mz_cuda_wzaes_ctr", i32, [vp, vp, vp, u32, u64, vp, u32, vp])
    sig("mz_cuda_wzaes_hmac", i32, [vp, vp, vp, u32, vp, u32, vp, vp])
    sig("mz_cuda_pkcrypt_workspace_bytes", u64, [u64, u32])
    sig("mz_cuda_pkcrypt_encrypt", i32, [vp, vp, vp, u32, C.c_char_p, vp, u64, vp])
    sig("mz_cuda_pkcrypt_decrypt", i32, [vp, vp, vp, u32, C.c_char_p, vp])
    sig("mz_cuda_gather_region_bound", u64, [u64])
    sig("mz_cuda_deflate_sharded", i32, [vp, i32, i32, i32, C.POINTER(u64), C.POINTER(u64), C.POINTER(u32)])
    sig("mz_cuda_ipc_export", i32, [vp, vp])
    sig("mz_cuda_ipc_open", i32, [vp, C.POINTER(vp)])
    sig("mz_cuda_ipc_close", i32, [vp])
    sig("mz_cuda_memcpy_peer", i32, [vp, vp, sz, vp])
    sig("mz_cuda_stream_wait_event", i32, [vp, vp])
    sig("mz_cuda_gather", i32, [vp, u64, vp, u32, vp, vp, vp])
    sig("mz_cuda_scatter_blobs", i32, [vp, vp, vp, u32, vp, vp])
    return L


class Shard(C.Structure):
    """mz_cuda_shard (include/mz_cuda_batch.h)"""
    _fields_ = [("device", C.c_int32), ("d_in", C.c_void_p), ("len", C.c_uint64), ("d_gathered", C.c_void_p), ("gathered_cap", C.c_uint64),
                ("d_rows", C.c_void_p)]


def check(err, what="call"):
    if err != MZ_OK:
        msg = load().mz_cuda_last_error()
        raise RuntimeError("%s failed: %d (%s)" % (what, err, msg.decode() if msg else ""))


def _stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class DeflateBatch:
    """Device-resident compression of one buffer cut into independent <=64 KiB chunks (K2+K3, K4, K1).

    Buffers are torch uint8 CUDA tensors; all work is enqueued on torch's current stream.
    """

    def __init__(self, max_bytes, chunk=CHUNK_MAX, with_crc=True):
        import torch
        self.lib = load()
        check(self.lib.mz_cuda_init(), "mz_cuda_init")
        self.chunk = chunk
        self.max_chunks = max(1, (max_bytes + chunk - 1) // chunk)
        self.stride = int(self.lib.mz_cuda_deflate_slot_bound(chunk))
        dev = torch.device("cuda", torch.cuda.current_device())
        self.slots = torch.empty(self.max_chunks * self.stride, dtype=torch.uint8, device=dev)
        self.out_len = torch.empty(self.max_chunks, dtype=torch.int32, device=dev)
        self.offsets = torch.empty(self.max_chunks + 1, dtype=torch.int64, device=dev)
        self.joined = torch.empty(self.max_chunks * self.stride, dtype=torch.uint8, device=dev)
        self.with_crc = with_crc
        if with_crc:
            self.residue = torch.empty(self.max_chunks, dtype=torch.int32, device=dev)
            self.chunk_crc = torch.empty(self.max_chunks, dtype=torch.int32, device=dev)
            self.crc_out = torch.empty(2, dtype=torch.int32, device=dev)

    def nchunks(self, nbytes):
        return max(1, (nbytes + self.chunk - 1) // self.chunk)

    def compress(self, src, nbytes, level=1, final=True, join=True, one_stream=False):
        """Enqueue K2+K3 (+K1 per-chunk CRC and fold) (+K4 join). Returns number of chunks."""
        n = self.nchunks(nbytes)
        assert n <= self.max_chunks and src.is_cuda and src.dtype.itemsize == 1
        s = _stream_ptr()
        check(self.lib.mz_cuda_deflate_chunks(src.data_ptr(), nbytes, self.chunk, None, None, None, n, (FLAG_FINAL if final else 0) | (FLAG_DICT if one_stream else 0),
                                              level, self.slots.data_ptr(), self.stride, self.out_len.data_ptr(), s), "deflate")
        if self.with_crc and nbytes > 0:
            check(self.lib.mz_cuda_crc32_segments(src.data_ptr(), nbytes, self.chunk, None, None, n, self.residue.data_ptr(),
                                                  self.chunk_crc.data_ptr(), s), "crc32")
            check(self.lib.mz_cuda_crc32_fold(self.residue.data_ptr(), n, self.chunk, nbytes, self.crc_out.data_ptr(), s), "crc fold")
        if join:
            check(self.lib.mz_cuda_concat(self.slots.data_ptr(), self.stride, self.out_len.data_ptr(), n, self.offsets.data_ptr(),
                                          self.joined.data_ptr(), s), "concat")
        return n

    def result(self, nchunks):
        """Synchronise and return (joined bytes as a CUDA tensor view, crc32 or None)."""
        import torch
        torch.cuda.current_stream().synchronize()
        total = int(self.offsets[nchunks].item())
        crc = (int(self.crc_out[1].item()) & 0xFFFFFFFF) if self.with_crc else None
        return self.joined[:total], crc


def crc32_device(tensor, nbytes=None, value=0):
    """mz_crypt_crc32_update over a CUDA tensor (K1)."""
    lib = load()
    out = C.c_uint32(0)
    n = tensor.numel() * tensor.element_size() if nbytes is None else nbytes
    check(lib.mz_cuda_crc32_device(tensor.data_ptr(), n, value, C.byref(out)), "crc32_device")
    return out.value


def inflate_device(comp, out_cap):
    """Decode ONE raw deflate stream held in a CUDA uint8 tensor (padded >=16 bytes). Returns (status, out tensor, consumed)."""
    import torch
    lib = load()
    dev = comp.device
    n = comp.numel()
    padded = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
    padded[:n] = comp
    out = torch.empty(out_cap + 512, dtype=torch.uint8, device=dev)
    job = InflateJob(padded.data_ptr(), 0, n, out.data_ptr(), 0, out_cap, 1, 0)
    st = InflateState()
    d_job = torch.frombuffer(bytearray(bytes(job)), dtype=torch.uint8).to(dev)
    d_st = torch.zeros(C.sizeof(InflateState), dtype=torch.uint8, device=dev)
    check(lib.mz_cuda_inflate_streams(d_job.data_ptr(), d_st.data_ptr(), 1, _stream_ptr()), "inflate")
    torch.cuda.current_stream().synchronize()
    raw = bytes(d_st.cpu().numpy().tobytes())
    C.memmove(C.byref(st), raw, C.sizeof(InflateState))
    return st.status, out[:st.out_pos], (st.in_bitpos + 7) // 8, st
