"""Scope row f4, PKWARE traditional encryption, on the device: K9's segmented encrypt and serial decrypt against the Python
restatement of APPNOTE 6.1, and whole PKWARE archives both ways against the reference built with mz_strm_pkcrypt.c -- the scenarios
of tests/test_emu_pkcrypt.py on the real library, with more and larger entries."""
import ctypes as C
import json
import os
import subprocess

import pytest

import pkcrypt_checks

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REFDIR = os.path.join(ROOT, "oracle", "_ref")


def _device_calls():
    import torch
    import __graft_entry__ as ge
    pkg = ge._load_pkg()
    lib = pkg.load()
    pkg.check(lib.mz_cuda_init())
    torch.cuda.set_device(0)
    tensors = {}

    def buf(b):
        t = torch.zeros(max(len(b), 1) + 16, dtype=torch.uint8, device="cuda")
        if len(b):
            t[:len(b)] = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        p = C.c_void_p(t.data_ptr())
        tensors[p.value] = t
        return p, t

    def back(p, n):
        torch.cuda.synchronize()
        return bytes(tensors[p.value][:n].cpu().numpy().tobytes())

    def call(name, *args):
        r = getattr(lib, name)(*args)
        torch.cuda.synchronize()
        return r
    return call, buf, back


@pytest.mark.gpu
def test_k9_known_answers_on_the_gpu(built):
    call, buf, back = _device_calls()
    pkcrypt_checks.run(call, buf, back, lens=(0, 1, 11, 12, 13, 4095, 4096, 4097, 65536, 70001, 1_000_003), big=5_000_017)


@pytest.mark.gpu
def test_k9_64mib_entry_segmented_encrypt_serial_decrypt(built):
    # the segmented encrypt of one 64 MiB entry, undone by the one-thread decrypt; the Python cipher checks the first 1 MiB
    call, buf, back = _device_calls()
    pkcrypt_checks.run(call, buf, back, lens=(), big=64 << 20, check_limit=1 << 20)


def _run_cmd(args, cwd, ok=True):
    r = subprocess.run([str(a) for a in args], cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
    if ok:
        assert r.returncode == 0, (args, r.returncode, r.stdout[-600:], r.stderr[-600:])
    return r


def _binaries():
    exe, refe = os.path.join(REFDIR, "zipbatch_cudae"), os.path.join(REFDIR, "minizip_refe")
    if not os.path.exists(exe) or not os.path.exists(refe):
        pytest.skip("oracle/_ref/zipbatch_cudae / minizip_refe not built (need the reference sources and OpenSSL headers at build time)")
    return exe, refe


@pytest.mark.gpu
def test_pkcrypt_archives_both_ways_on_the_gpu(built, tmp_path):
    exe, refe = _binaries()
    pkcrypt_checks.pk_roundtrip(exe, refe, tmp_path, _run_cmd, n=2500, esz=65536)


@pytest.mark.gpu
def test_pkcrypt_single_256mib_entry_read_by_the_reference(built, tmp_path):
    exe, refe = _binaries()
    shim = pkcrypt_checks.build_shim(tmp_path)
    (tmp_path / "dump").mkdir()
    cmd = pkcrypt_checks.driver_cmd(exe, shim, ["big.zip", 1, 256 << 20, 6, "native_pk", "dump", 1])
    st = json.loads(_run_cmd(cmd, tmp_path).stdout.decode().strip().splitlines()[-1])
    assert st["err"] == 0 and st["entries"] == 1 and st["bytes_in"] == 256 << 20
    _run_cmd([refe, "-x", "-o", "-p", "secret", "-d", "out", "big.zip"], tmp_path)
    assert (tmp_path / "out" / "e" / "000000").read_bytes() == (tmp_path / "dump" / "000000").read_bytes()
