"""Shared checks for K9 (PKWARE traditional encryption, scope row f4): an independent restatement of the cipher from APPNOTE 6.1.5-6.1.6
in Python, known answers for odd lengths, unaligned offsets and several passwords, then whole archives both ways against the reference
built with mz_strm_pkcrypt.c (oracle/_ref/minizip_refe) and against Python's zipfile as a second reader.
`call(name, *args)` invokes the product entry point; `buf(bytes)` gives (pointer, keepalive) for device-visible memory and `back(ptr, n)`
reads it back."""
import json
import os
import zipfile
import zlib

_TAB = []
for _i in range(256):
    _r = _i
    for _ in range(8):
        _r = (_r >> 1) ^ (0xEDB88320 if _r & 1 else 0)
    _TAB.append(_r)


class Cipher:
    """APPNOTE 6.1.5: three keys; 6.1.6: the key stream byte is taken from key2 before the plain byte updates the keys."""

    def __init__(self, password):
        self.k0, self.k1, self.k2 = 305419896, 591751049, 878082192
        for b in password:
            self._update(b)

    def _update(self, b):
        self.k0 = _TAB[(self.k0 ^ b) & 0xFF] ^ (self.k0 >> 8)
        self.k1 = ((self.k1 + (self.k0 & 0xFF)) * 134775813 + 1) & 0xFFFFFFFF
        self.k2 = _TAB[(self.k2 ^ (self.k1 >> 24)) & 0xFF] ^ (self.k2 >> 8)

    def _stream(self):
        t = (self.k2 | 2) & 0xFFFF
        return ((t * (t ^ 1)) >> 8) & 0xFF

    def encrypt(self, data):
        out = bytearray(len(data))
        for i, b in enumerate(data):
            out[i] = b ^ self._stream()
            self._update(b)
        return bytes(out)

    def decrypt(self, data):
        out = bytearray(len(data))
        for i, c in enumerate(data):
            b = c ^ self._stream()
            out[i] = b
            self._update(b)
        return bytes(out)


PASSWORDS = (b"", bytes((33 + i % 90) for i in range(200)), "pässwörd-秘密".encode("utf-8"))


def run(call, buf, back, lens=(0, 1, 11, 12, 13, 4095, 4096, 4097, 70001), big=600_001, check_limit=None):
    """Encrypt a batch (the given lengths plus one entry of `big` bytes spanning many segments) at unaligned offsets with five bytes
    of guard between entries, compare with the Python cipher (the first check_limit bytes of each entry when given), decrypt and
    compare with the plaintext."""
    lens = tuple(lens) + (big,)
    n = len(lens)
    offs, pos = [], 3
    for ln in lens:
        offs.append(pos)
        pos += ln + 5
    plain = os.urandom(pos)
    for pw in PASSWORDS:
        p_data, k1 = buf(plain)
        p_off, k2 = buf(b"".join(o.to_bytes(8, "little") for o in offs))
        p_len, k3 = buf(b"".join(ln.to_bytes(8, "little") for ln in lens))
        wsb = call("mz_cuda_pkcrypt_workspace_bytes", sum(lens), n)
        p_ws, k4 = buf(bytes(wsb))
        assert call("mz_cuda_pkcrypt_encrypt", p_data, p_off, p_len, n, pw, p_ws, wsb, None) == 0
        data = back(p_data, pos)
        for e in range(n):
            m = lens[e] if check_limit is None else min(lens[e], check_limit)
            assert data[offs[e]:offs[e] + m] == Cipher(pw).encrypt(plain[offs[e]:offs[e] + m]), (pw, e, lens[e], "encrypt")
            end = offs[e] + lens[e]
            assert data[end:end + 5] == plain[end:end + 5]  # bytes between the entries are not touched
        assert data[:3] == plain[:3]
        assert call("mz_cuda_pkcrypt_decrypt", p_data, p_off, p_len, n, pw, None) == 0
        assert back(p_data, pos) == plain, (pw, "decrypt(encrypt(x)) != x")
    # an empty batch; parameter errors (MZ_PARAM_ERROR = -102)
    p_ws, k5 = buf(bytes(256))
    assert call("mz_cuda_pkcrypt_encrypt", None, None, None, 0, b"pw", p_ws, 256, None) == 0
    assert call("mz_cuda_pkcrypt_decrypt", None, None, None, 0, b"pw", None) == 0
    p_data, k1 = buf(plain)
    p_off, k2 = buf(b"".join(o.to_bytes(8, "little") for o in offs))
    p_len, k3 = buf(b"".join(ln.to_bytes(8, "little") for ln in lens))
    assert call("mz_cuda_pkcrypt_encrypt", p_data, p_off, p_len, n, None, p_ws, 256, None) == -102
    assert call("mz_cuda_pkcrypt_decrypt", p_data, p_off, p_len, n, None, None) == -102
    assert call("mz_cuda_pkcrypt_encrypt", p_data, p_off, p_len, n, b"pw", p_ws, 256, None) == -102  # workspace too small
    assert back(p_data, pos) == plain  # refused calls leave the data alone


def _last_json(r):
    return json.loads(r.stdout.decode().strip().splitlines()[-1])


def _inflate_exact(stream):
    d = zlib.decompressobj(-15)
    out = d.decompress(stream)
    assert d.eof and d.unused_data == b"", "the stored size is not stream + 12"
    return out


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the C4 driver's modes for the PKWARE entry points: its AES modes with tests/support/zipbatch_pkshim.c preloaded (True), or as they are
PK_MODES = {"native_pk": ("native_aes", True), "native_pk_sha": ("native_aes_sha", True), "extract_pk": ("extract_aes", True),
            "extract_ref_pk": ("extract_ref_aes", False)}


def build_shim(out_dir):
    """compile tests/support/zipbatch_pkshim.c (the project's headers only) into out_dir; returns its path"""
    import subprocess
    so = os.path.join(str(out_dir), "libzbpkshim.so")
    r = subprocess.run(["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-o", so,
                        os.path.join(ROOT, "tests", "support", "zipbatch_pkshim.c"), "-ldl"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-2000:]
    return so


def driver_cmd(exe, shim, args, password=None):
    """the driver's command line for args = [archive, entries, entry_bytes, level, mode, ...] with PKWARE modes mapped"""
    mode, pre = PK_MODES.get(args[4], (args[4], False))
    env = ["env"] + (["LD_PRELOAD=" + shim] if pre else []) + (["ZIPBATCH_PASSWORD=" + password] if password else [])
    return env + [exe] + [str(a) for a in args[:4]] + [mode] + [str(a) for a in args[5:]]


def pk_roundtrip(exe_e, refe, tmp_path, run_cmd, n=60, esz=30_000):
    """archives both ways: ours (native writer + K9) -> the reference CLI and Python's zipfile extract with the password; the
    reference's own PKWARE archive (data descriptors, time-based verifier) -> the batch extractor; wrong password, damaged ciphertext
    and the AES-only extractor are refused with the reference's codes; an AES archive reads through the new entry point."""
    shim = build_shim(tmp_path)

    def zb(args, password=None, ok=True):
        return _last_json(run_cmd(driver_cmd(exe_e, shim, args, password), tmp_path, ok=ok))
    (tmp_path / "dump").mkdir()
    st = zb(["p.zip", str(n), str(esz), "6", "native_pk", "dump", "7"])
    assert st["err"] == 0 and st["entries"] == n
    with zipfile.ZipFile(tmp_path / "p.zip") as z:
        infos = z.infolist()
        for i in infos:
            assert i.flag_bits & 0x809 == 0x801 and i.compress_type == 8 and i.extract_version == 20, (i.filename, i.flag_bits, i.extract_version)
        raw = (tmp_path / "p.zip").read_bytes()
        for k in range(0, n, 7):
            i = infos[k]
            want = (tmp_path / "dump" / ("%06d" % k)).read_bytes()
            assert z.read(i, pwd=b"secret") == want  # a second, independent reader
            start = i.header_offset + 30 + len(i.filename.encode()) + len(i.extra)
            plain = Cipher(b"secret").decrypt(raw[start:start + i.compress_size])
            assert plain[11] == (i.CRC >> 24) & 0xFF and plain[10] == (i.CRC >> 16) & 0xFF
            assert _inflate_exact(plain[12:]) == want  # stored size = stream + 12
    run_cmd([refe, "-x", "-o", "-p", "secret", "-d", "outp", "p.zip"], tmp_path)
    for k in range(0, n, 7):
        assert (tmp_path / "outp" / "e" / ("%06d" % k)).read_bytes() == (tmp_path / "dump" / ("%06d" % k)).read_bytes()
    got = zb(["p.zip", str(n), str(esz), "0", "extract_pk"])
    want = zb(["p.zip", str(n), str(esz), "0", "extract_ref_pk"])
    assert got["err"] == 0 and want["err"] == 0 and got["entries"] == want["entries"] == n and got["bytes_out"] == want["bytes_out"]
    assert got["mismatches"] == 0 and got["verified"] > 0
    bad = zb(["p.zip", str(n), str(esz), "0", "extract_pk"], password="wrong", ok=False)
    assert bad["err"] == -108  # MZ_PASSWORD_ERROR
    # the AES-only extractor keeps its contract
    old = zb(["p.zip", str(n), str(esz), "0", "extract_aes"], ok=False)
    assert old["err"] == -109  # MZ_SUPPORT_ERROR
    # one flipped ciphertext bit inside an incompressible entry's stored block: PKWARE has no MAC, the CRC catches it
    victim = infos[9]
    start = victim.header_offset + 30 + len(victim.filename.encode()) + len(victim.extra)
    damaged = bytearray(raw)
    damaged[start + 12 + 100] ^= 1
    (tmp_path / "p_bad.zip").write_bytes(bytes(damaged))
    bad = zb(["p_bad.zip", str(n), str(esz), "0", "extract_pk"], ok=False)
    assert bad["err"] in (-105, -3), bad  # MZ_CRC_ERROR, MZ_DATA_ERROR
    # with SHA-256 extra fields: the reference verifies them on extraction
    (tmp_path / "dumps").mkdir()
    st = zb(["ps.zip", str(n), str(esz), "6", "native_pk_sha", "dumps", "5"])
    assert st["err"] == 0
    run_cmd([refe, "-x", "-o", "-p", "secret", "-d", "outs", "ps.zip"], tmp_path)
    for k in range(0, n, 5):
        assert (tmp_path / "outs" / "e" / ("%06d" % k)).read_bytes() == (tmp_path / "dumps" / ("%06d" % k)).read_bytes()
    got = zb(["ps.zip", str(n), str(esz), "0", "extract_pk"])
    assert got["err"] == 0 and got["entries"] == n and got["mismatches"] == 0
    # an archive the REFERENCE encrypted: data descriptors and the time-based verifier (flag 0x809), an empty entry (14 stored bytes)
    src = tmp_path / "src"
    src.mkdir()
    files = {"t1.txt": b"the quick brown fox " * 9000, "t2.bin": os.urandom(3000), "empty.bin": b""}
    for k, v in files.items():
        (src / k).write_bytes(v)
    run_cmd([refe, "-p", "secret", "-o", "../r_p.zip"] + sorted(files), src)
    with zipfile.ZipFile(tmp_path / "r_p.zip") as z:
        for i in z.infolist():
            assert i.flag_bits & 0x809 == 0x809, i.flag_bits
            if i.filename == "empty.bin":
                assert i.compress_size == 14
    got = zb(["r_p.zip", "3", str(1 << 20), "0", "extract_pk"])
    assert got["err"] == 0 and got["entries"] == 3 and got["bytes_out"] == sum(len(v) for v in files.values())
    bad = zb(["r_p.zip", "3", str(1 << 20), "0", "extract_pk"], password="wrong", ok=False)
    assert bad["err"] == -108
    # plain and WinZip AES archives read through the same entry point
    st = zb(["a.zip", str(n), str(esz), "6", "native_aes"])
    assert st["err"] == 0
    got = zb(["a.zip", str(n), str(esz), "0", "extract_pk"])
    assert got["err"] == 0 and got["entries"] == n and got["mismatches"] == 0
    st = zb(["plain.zip", str(n), str(esz), "6", "native"])
    assert st["err"] == 0
    got = zb(["plain.zip", str(n), str(esz), "0", "extract_pk"])
    assert got["err"] == 0 and got["entries"] == n and got["mismatches"] == 0
