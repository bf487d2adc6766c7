#!/usr/bin/env python3
"""K9 (PKWARE traditional encryption) on one GPU, device-resident, CUDA events over warmed repeated launches:
  - the segmented encrypt of 4096 x 64 KiB and of 1 x 256 MiB (the same bytes; the time must follow the bytes, not the largest entry),
    for each segment size in MZ_CUDA_PKCRYPT_SEG's range;
  - the one-thread-per-entry decrypt of 1 x 16 MiB (the per-thread rate) and of 4096 x 64 KiB (aggregate);
  - optionally (--zip) the native writer: zipbatch_cudae ENTRIES 65536 6, PKWARE (its native_aes mode with
    tests/support/zipbatch_pkshim.c preloaded) against native, alternating, archives in a temporary directory.
The multi-entry encrypt is checked by decrypting it again. Prints the card's name and power limit, then one JSON line per measurement.
usage: bench_pkcrypt.py [--zip] [--entries N]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import __graft_entry__ as ge  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--zip", action="store_true", help="also time the native writer (zipbatch_cudae)")
    ap.add_argument("--entries", type=int, default=100000)
    a = ap.parse_args()
    pkg = ge._load_pkg()
    lib = pkg.load()
    pkg.check(lib.mz_cuda_init())
    torch.cuda.set_device(0)
    print(json.dumps({"card": card(), "torch": torch.__version__}), flush=True)
    total = 256 << 20
    data = torch.randint(0, 256, (total + 64,), dtype=torch.uint8, device="cuda")
    keep = data.clone()
    pw = b"secret"
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def layout(n, size):
        off = torch.arange(n, dtype=torch.int64, device="cuda") * size
        ln = torch.full((n,), size, dtype=torch.int64, device="cuda")
        return off, ln

    def timed(fn, reps):
        fn()
        fn()
        torch.cuda.synchronize()
        ev[0].record()
        for _ in range(reps):
            fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / reps

    def check_roundtrip(n, off, ln, nbytes):
        data.copy_(keep)
        ws = int(lib.mz_cuda_pkcrypt_workspace_bytes(nbytes, n))
        w = torch.empty(ws, dtype=torch.uint8, device="cuda")
        pkg.check(lib.mz_cuda_pkcrypt_encrypt(data.data_ptr(), off.data_ptr(), ln.data_ptr(), n, pw, w.data_ptr(), ws, None), "encrypt")
        changed = not torch.equal(data[:nbytes], keep[:nbytes])
        pkg.check(lib.mz_cuda_pkcrypt_decrypt(data.data_ptr(), off.data_ptr(), ln.data_ptr(), n, pw, None), "decrypt")
        torch.cuda.synchronize()
        return changed and torch.equal(data, keep)

    shapes = {"4096x64KiB": (4096, 65536), "1x256MiB": (1, total)}
    for seg in (256, 512, 1024, 2048, 4096):
        os.environ["MZ_CUDA_PKCRYPT_SEG"] = str(seg)
        row = {"what": "pkcrypt_encrypt", "seg": seg}
        for name, (n, size) in shapes.items():
            off, ln = layout(n, size)
            ws = int(lib.mz_cuda_pkcrypt_workspace_bytes(total, n))
            w = torch.empty(ws, dtype=torch.uint8, device="cuda")
            ms = timed(lambda: pkg.check(lib.mz_cuda_pkcrypt_encrypt(data.data_ptr(), off.data_ptr(), ln.data_ptr(), n, pw, w.data_ptr(), ws, None)), 10)
            row[name + "_ms"] = round(ms, 3)
            row[name + "_GBps"] = round(total / ms / 1e6, 2)
            if n > 1:  # (the 256 MiB entry's round trip is one thread decrypting for seconds: tests/test_gpu_pkcrypt.py covers it)
                row[name + "_roundtrip_ok"] = check_roundtrip(n, off, ln, total)
        row["ratio_1x256MiB_over_4096x64KiB"] = round(row["1x256MiB_ms"] / row["4096x64KiB_ms"], 3)
        print(json.dumps(row), flush=True)
    os.environ.pop("MZ_CUDA_PKCRYPT_SEG")
    for name, (n, size), reps in (("1x16MiB", (1, 16 << 20), 3), ("4096x64KiB", (4096, 65536), 3)):
        off, ln = layout(n, size)
        ms = timed(lambda: pkg.check(lib.mz_cuda_pkcrypt_decrypt(data.data_ptr(), off.data_ptr(), ln.data_ptr(), n, pw, None)), reps)
        nbytes = n * size
        print(json.dumps({"what": "pkcrypt_decrypt", "shape": name, "ms": round(ms, 3), "MBps_per_thread": round(size / ms / 1e3, 2),
                          "GBps_aggregate": round(nbytes / ms / 1e6, 3)}), flush=True)
    if a.zip:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import pkcrypt_checks
        exe = os.path.join(ROOT, "oracle", "_ref", "zipbatch_cudae")
        shimdir = tempfile.mkdtemp()
        shim = pkcrypt_checks.build_shim(shimdir)
        for rep in range(2):
            for mode in ("native", "native_pk"):
                with tempfile.TemporaryDirectory() as d:
                    cmd = pkcrypt_checks.driver_cmd(exe, shim, [os.path.join(d, "c4.zip"), a.entries, 65536, 6, mode])
                    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=dict(os.environ, ZIPBATCH_REPEAT="3"))
                    for line in r.stdout.strip().splitlines():
                        row = json.loads(line)
                        row["what"] = "zipbatch"
                        row["pass"] = rep
                        row["mode"] = mode
                        print(json.dumps(row), flush=True)
                    if r.returncode:
                        print(json.dumps({"what": "zipbatch", "mode": mode, "rc": r.returncode, "stderr": r.stderr[-400:]}), flush=True)


if __name__ == "__main__":
    main()
