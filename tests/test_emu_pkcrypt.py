"""Scope row f4, PKWARE traditional encryption, on the CPU: K9 (minizip-ng_b200/csrc/pkcrypt_kernel.cuh) run on the execution-model
emulator against the Python restatement of APPNOTE 6.1, with small segments so that the carries cross many tiles; then whole PKWARE
archives both ways against the reference built with its mz_strm_pkcrypt.c (oracle/_ref/minizip_refe)."""
import ctypes as C
import os
import subprocess

import pytest

import pkcrypt_checks

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REFDIR = os.path.join(ROOT, "oracle", "_ref")


@pytest.fixture(scope="module")
def emuprod():
    r = subprocess.run(["make", "-s", "-C", os.path.join(HERE, "emu"), "libmz_strm_emu.so"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]
    import cuharness
    return cuharness.pkg().configure(C.CDLL(os.path.join(HERE, "emu", "libmz_strm_emu.so")))


def _host_calls(lib):
    def buf(b):
        m = C.create_string_buffer(bytes(b), max(len(b), 1))
        return C.cast(m, C.c_void_p), m

    def back(p, n):
        return C.string_at(p, n)

    def call(name, *args):
        return getattr(lib, name)(*args)
    return call, buf, back


@pytest.mark.parametrize("seg", [None, "256"])
def test_k9_known_answers_on_the_emulator(emuprod, monkeypatch, seg):
    # MZ_CUDA_PKCRYPT_SEG=256: the 600 KB entry is ~2300 segments, nine tiles, so the carry crosses tiles of the pass kernels
    if seg:
        monkeypatch.setenv("MZ_CUDA_PKCRYPT_SEG", seg)
    call, buf, back = _host_calls(emuprod)
    pkcrypt_checks.run(call, buf, back)


def test_pkcrypt_archives_both_ways_against_the_reference(emuprod, tmp_path):
    if not os.path.exists("/usr/include/openssl/sha.h"):
        pytest.skip("needs the OpenSSL headers (the reference's crypto provider)")
    r = subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "_ref/minizip_refe", "_ref/zipbatch_emue"], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0 and "No rule to make target" in r.stdout:
        pytest.skip("the reference's sources are absent (oracle/Makefile REF)")
    assert r.returncode == 0, r.stdout[-3000:]

    def run_cmd(args, cwd, ok=True):
        r = subprocess.run([str(a) for a in args], cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
        if ok:
            assert r.returncode == 0, (args, r.returncode, r.stdout[-600:], r.stderr[-600:])
        return r
    pkcrypt_checks.pk_roundtrip(os.path.join(REFDIR, "zipbatch_emue"), os.path.join(REFDIR, "minizip_refe"), tmp_path, run_cmd)
