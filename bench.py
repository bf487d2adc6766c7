#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 DEFLATE + CRC-32 backend (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (mz_strm_zlib over zlib 1.3)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as .npy files

Workload (config C5, `configs[4]`, the configuration the metric is quoted on): a 16 GiB synthetic enwik-style
buffer, cut into independent 64 KiB chunks, DEFLATE level 1 + per-chunk CRC-32 + CRC fold + join (K2+K3, K1, K4).
A step = one pass over the whole buffer. With N GPUs the SAME 16 GiB is sharded by contiguous chunk ranges
(strong scaling), each rank compresses its shard, and one NCCL all-gather returns every rank's joined bitstream
and per-chunk {crc, length} table.

value      whole-job GiB/s of uncompressed input, inputs resident in HBM, CUDA-event timed, max over ranks
e2e        same metric through the reference-facing vtbl call (mz_stream_cuda_write/close) with HOST buffers:
           pinned host input, host->device copies, device->host of the stream, base-stream sink, all timed
roofline   dominant kernel (deflate_chunks_kernel): algorithmic bytes (input bytes read per launch) / mean launch time
           (CUDA events on the launching stream) vs the measured HBM copy bandwidth (MEASURED_PEAKS.json)
cpu_baseline the reference path (oracle/_ref: mz_strm_zlib.c + mz_crypt.c + zlib 1.3) on the host cores, bounded sample
"""
import argparse
import ctypes as C
import faulthandler
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GiB = 1 << 30
METRIC = "deflate_l1_crc32_input_throughput"
UNIT = "GiB/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c5", choices=["c1", "c2", "c3", "c4", "c5"],
                    help="BASELINE.json configs[0..4]; c5 (default) is the configuration the metric is quoted on")
    ap.add_argument("--size-gib", type=float, default=None, help="override the configuration's size (c5: 16 GiB, c3: 4 GiB, c2: 0.25 GiB)")
    ap.add_argument("--level", type=int, default=1)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-sample-mib", type=int, default=2048)
    ap.add_argument("--sub-batches", type=int, default=0, help="pieces per shard when N>1 (all-gather of piece j overlaps compression of j+1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (config c5 only; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != "c5" or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of config c5, --impl ours")
    if args.size_gib is None:
        args.size_gib = {"c1": 0.0625, "c2": 0.25, "c3": 4.0, "c4": 100000 * 65536 / GiB, "c5": 16.0}[args.config]
    if args.config == "c2" and "--level" not in " ".join(sys.argv):
        args.level = 6
    if args.config == "c4" and "--level" not in " ".join(sys.argv):
        args.level = 6
    return args


def usable_cores():
    """Host threads this process may really use: the scheduler affinity mask capped by the cgroup CPU quota (os.cpu_count()
    reports the machine, not the lease). Returns (cores, details)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    cores = aff if quota is None else max(1, min(aff, int(quota)))
    return cores, {"affinity": aff, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


# ---- clocks --------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled every few milliseconds from a thread
    (a multi-GPU step is tens of milliseconds, too short for `nvidia-smi -lms`); falls back to nvidia-smi when the
    NVML bindings are missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None
        self.thread = None
        self.samples = []
        self.mask = 0
        self.max_mhz = None
        self.stop_flag = False

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)

    def _poll(self, nv, h):
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        try:
            import threading
            nv, h = self._nvml_handle()
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread:
            self.stop_flag = True
            self.thread.join(timeout=2)
            sm = sorted(self.samples)
            reasons = sorted(name for bit, name in self.REASONS if self.mask & bit)
            return {"sm_mhz": float(sm[len(sm) // 2]) if sm else None, "sm_max_mhz": float(self.max_mhz) if self.max_mhz else None, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        except Exception:
            pass
        finally:
            try:
                os.unlink(self.path)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi"}


# ---- the reference's CPU path (oracle/_ref) -------------------------------------------------------------------------
def cpu_reference_throughput(sample, level, threads=None, window_bits=-15, piece=None):
    """Time mz_stream_zlib (level `level`) + mz_crypt_crc32_update over `sample` (bytes) split across host threads.
    Each thread drives the reference's own loop mz_stream_copy_stream_to_end (mz_strm.c:191-206: 16 KiB writes) into a
    reference memory stream, one independent stream per piece (4..32 MiB, or `piece`). Returns (GiB/s, threads, compressed_bytes)."""
    import refshim
    ref = refshim.RefLib()
    n = len(sample)
    threads = threads or usable_cores()[0]
    piece = piece or max(4 << 20, min(32 << 20, (n // (threads * 4)) >> 20 << 20))
    jobs = [(o, min(piece, n - o)) for o in range(0, n, piece)]
    base = C.addressof(sample)
    lock = threading.Lock()
    state = {"next": 0, "comp": 0, "err": 0}

    def work():
        L = ref.lib
        while True:
            with lock:
                i = state["next"]
                state["next"] += 1
            if i >= len(jobs):
                return
            off, ln = jobs[i]
            src = L.mz_stream_mem_create()
            L.mz_stream_mem_set_buffer(src, base + off, ln)
            L.mz_stream_open(src, None, refshim.MZ_OPEN_MODE_READ)
            sink = ref.mem_sink(grow=8 << 20)
            z = L.mz_stream_zlib_create()
            L.mz_stream_set_prop_int64(z, refshim.PROP_COMPRESS_LEVEL, level)
            L.mz_stream_set_prop_int64(z, refshim.PROP_COMPRESS_WINDOW, window_bits)
            L.mz_stream_set_base(z, sink)
            ok = L.mz_stream_open(z, None, refshim.MZ_OPEN_MODE_WRITE) == 0
            ok = ok and L.mz_stream_copy_stream_to_end(z, None, src, None) == 0
            L.mz_stream_close(z)
            crc = L.mz_crypt_crc32_update(0, base + off, ln)  # the CRC the zip path computes beside the codec (mz_zip.c:2064)
            tout = ref.get_prop(z, refshim.PROP_TOTAL_OUT)[1]
            ref.delete(z)
            L.mz_stream_close(sink)
            ref.delete(sink)
            ref.delete(src)
            with lock:
                state["comp"] += tout
                if not ok or crc is None:
                    state["err"] += 1

    t0 = time.perf_counter()
    ts = [threading.Thread(target=work) for _ in range(min(threads, len(jobs)))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    dt = time.perf_counter() - t0
    assert state["err"] == 0
    return n / GiB / dt, len(ts), state["comp"]


def host_text_sample(nbytes, seed=99):
    """The bench text from the HOST generator (tests/support/textgen_host.c via libmztest.so): the reference arm never loads the
    GPU library, and the bytes are the same as the device generator's for the same seed."""
    import textgen
    return textgen.host_buffer(nbytes, seed)


WORKLOADS = {
    "c1": "C1: CRC-32 of a 64 MiB buffer via mz_crypt_crc32_update",
    "c2": "C2: minigzip-style deflate level %(level)d (gzip framing) of a %(mib)d MiB synthetic text buffer, one stream (64 KiB chunks that may refer back 32 KiB: MZ_CUDA_FLAG_DICT)",
    "c3": "C3: inflate one %(gib).2f GiB multi-block .gz member (zlib level 6 blocks) through the stream read() call",
    "c4": "C4: zip of %(entries)d x 64 KiB entries, per-entry deflate level %(level)d + CRC-32",
    "c5": "C5: %(gib).2f GiB enwik-style buffer, independent 64 KiB chunks, DEFLATE level %(level)d + CRC-32 per chunk + fold + join",
}
METRICS = {"c1": ("crc32_input_throughput", "GiB/s"), "c2": ("gzip_l6_input_throughput", "GiB/s"), "c3": ("inflate_output_throughput", "GiB/s"),
           "c4": ("zip_deflate_crc_input_throughput", "GiB/s"), "c5": (METRIC, UNIT)}
REF_PATH = "mz_strm_zlib.c + mz_crypt.c over system zlib 1.3 (zlib-ng is not vendored / not buildable offline)"


def workload_text(args):
    return WORKLOADS[args.config] % {"level": args.level, "mib": int(args.size_gib * 1024), "gib": args.size_gib,
                                     "entries": int(round(args.size_gib * GiB / 65536))}


def make_gzip_member(text_buf, nbytes, level=6, threads=None, piece=64 << 20):
    """One gzip member over text_buf[0..nbytes), made by zlib itself (CPython's zlib = the system zlib 1.3 the reference links):
    pieces are deflated in parallel, every piece but the last ends with Z_SYNC_FLUSH, so the concatenation is ONE valid raw
    stream of ordinary zlib blocks (no history across pieces); CRC-32 and ISIZE (mod 2^32) in the trailer. Building a 4 GiB
    member with one zlib stream would take minutes of single-core time."""
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    mv = memoryview(text_buf).cast("B")[:nbytes]
    offs = list(range(0, nbytes, piece))

    def one(o):
        last = o + piece >= nbytes
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        return co.compress(mv[o:o + piece]) + (co.flush(zlib.Z_FINISH) if last else co.flush(zlib.Z_SYNC_FLUSH))

    with ThreadPoolExecutor(max_workers=threads or usable_cores()[0]) as ex:
        parts = list(ex.map(one, offs))
    crc = 0
    for o in offs:
        crc = zlib.crc32(mv[o:o + piece], crc)
    hdr = bytes([0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 3])
    return hdr + b"".join(parts) + (crc & 0xffffffff).to_bytes(4, "little") + (nbytes & 0xffffffff).to_bytes(4, "little"), crc & 0xffffffff


def ref_line(args, value, ms, steps, cores, cores_info, sample, extra=None):
    metric, unit = METRICS[args.config]
    line = {
        "impl": "reference", "metric": metric, "value": round(value, 4), "unit": unit, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_text(args), "reference_path": REF_PATH, "sample": sample, "host_cores": cores_info},
        "cpu_baseline": {"value": round(value, 4), "unit": unit, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": round(value, 4), "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if extra:
        line.update(extra)
    print(json.dumps(line), flush=True)


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the configuration's path (oracle/_ref = the reference's sources compiled where
    they lie + zlib 1.3), on the host cores this process may use. Loads only oracle/_ref and tests/support/libmztest.so."""
    if rank != 0:
        return
    import refshim
    if not refshim.ref_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmzref.so missing (reference sources were not present at build time)"}))
        return
    cores, cinfo = usable_cores()
    ref = refshim.RefLib()
    cfg = args.config
    if cfg == "c5" or cfg == "c2":
        # the all-core figure: one independent stream per piece (the reference is single-threaded; this is the upper bound a
        # caller could get by running one reference stream per core), plus the single-stream figure the reference itself delivers
        nbytes = (args.cpu_sample_mib << 20) if cfg == "c5" else min(int(args.size_gib * GiB), 256 << 20)
        wb = -15 if cfg == "c5" else 31
        sample = host_text_sample(nbytes)
        vals = []
        for i in range(args.warmup + args.steps):
            v, thr, comp = cpu_reference_throughput(sample, args.level, threads=cores, window_bits=wb)
            if i >= args.warmup:
                vals.append(v)
            if i == 0 and nbytes / GiB / v > 60:  # keep the whole arm within a few minutes
                break
        vals = vals or [v]
        value = sum(vals) / len(vals)
        one_n = min(nbytes, 32 << 20)
        one = (C.c_uint8 * one_n).from_buffer(sample)
        v1, _, _ = cpu_reference_throughput(one, args.level, threads=1, window_bits=wb, piece=one_n)
        ref_line(args, value, 1000 * nbytes / GiB / value, len(vals), thr, cinfo,
                 "%d MiB of the bench text per step, one independent mz_stream_zlib (level %d, window bits %d) per 4..32 MiB piece on %d host threads, "
                 "+ mz_crypt_crc32_update per piece" % (nbytes >> 20, args.level, wb, thr),
                 {"ratio": round(comp / nbytes, 4), "single_stream": {"value": round(v1, 4), "unit": "GiB/s", "cores": 1,
                                                                      "sample": "one mz_stream_zlib over %d MiB: what one reference stream delivers" % (one_n >> 20)}})
    elif cfg == "c1":
        import numpy as np
        n = 64 << 20
        data = np.random.default_rng(1).integers(0, 256, n, dtype=np.uint8)
        vals = []
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            crc = ref.lib.mz_crypt_crc32_update(0, data.ctypes.data, n)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                vals.append(n / GiB / dt)
        value = sum(vals) / len(vals)
        ref_line(args, value, 1000 * n / GiB / value, len(vals), 1, cinfo, "one mz_crypt_crc32_update call over the 64 MiB buffer (zlib crc32), one core: the function is single-threaded",
                 {"crc32": "%08x" % (crc & 0xffffffff)})
    elif cfg == "c3":
        nbytes = min(int(args.size_gib * GiB), 1 << 30)  # bounded sample: one core inflates ~0.25 GB/s
        text = host_text_sample(nbytes)
        member, crc = make_gzip_member(text, nbytes, 6, cores)
        vals = []
        for i in range(min(args.warmup, 1) + min(args.steps, 3)):
            t0 = time.perf_counter()
            out = ref.zlib_decompress(member, window_bits=31, read_size=1 << 16)
            dt = time.perf_counter() - t0
            assert len(out) == nbytes
            if i >= min(args.warmup, 1):
                vals.append(nbytes / GiB / dt)
        value = sum(vals) / len(vals)
        ref_line(args, value, 1000 * nbytes / GiB / value, len(vals), 1, cinfo,
                 "one %d MiB gzip member of the bench text (zlib level 6 blocks) read through mz_stream_zlib_read in 64 KiB calls, one core: "
                 "a single member cannot be split across cores by the reference" % (nbytes >> 20), {"ratio": round(len(member) / nbytes, 4)})
    elif cfg == "c4":
        exe = os.path.join(ROOT, "oracle", "_ref", "zipbatch_ref")
        if not os.path.exists(exe):
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/zipbatch_ref missing"}))
            return
        entries = 6000  # bounded sample: ~0.8 k entries/s on one core
        d = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        vals = []
        try:
            for i in range(min(args.warmup, 1) + min(args.steps, 3)):
                r = subprocess.run([exe, os.path.join(d, "r.zip"), str(entries), "65536", str(args.level), "ref"], stdout=subprocess.PIPE, text=True, timeout=600)
                j = json.loads(r.stdout.strip().splitlines()[-1])
                assert j["err"] == 0 and j["close_err"] == 0
                if i >= min(args.warmup, 1):
                    vals.append(j)
        finally:
            subprocess.run(["rm", "-rf", d])
        value = sum(v["GiB_per_s"] for v in vals) / len(vals)
        eps = sum(v["entries_per_s"] for v in vals) / len(vals)
        ref_line(args, value, 1000 * (entries * 65536 / GiB) / max(value, 1e-9), len(vals), 1, cinfo,
                 "%d entries x 64 KiB through mz_zip_entry_write_open(raw=0)/write/close (mz_stream_zlib level %d + mz_crypt_crc32_update), archive on tmpfs, "
                 "one core: the reference's zip writer is single-threaded" % (entries, args.level), {"entries_per_s": round(eps, 1)})


# ---- our arm ---------------------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 22  # stream bytes --dump-outputs keeps over all ranks: 16 MiB as float32 plus 32 MiB of float64 positions


def dump_outputs(out_dir, rank, world, lib, pkg, dev, nbytes, crc, stream, stream_len, crc_rows, len_rows):
    """--dump-outputs (config c5): what a caller of the timed path receives from its last step, as DIR/<name>.npy --
    chunk_crc32 and chunk_compressed_bytes (one row per 64 KiB chunk), totals = [input bytes, stream bytes, CRC-32 of the
    input], and stream_sample = bytes of the joined DEFLATE stream at the sorted positions stream_sample_positions (seed 0;
    every position when the stream is that short). float64 holds every uint32 exactly, float32 every byte. With N GPUs each
    rank writes its own shard's arrays with the suffix _rank<r>."""
    import numpy as np
    import torch
    n = nbytes // 65536
    rows = torch.empty(2 * n, dtype=torch.int32, device=dev)
    pkg.check(lib.mz_cuda_memcpy_d2d(rows.data_ptr(), crc_rows, 4 * n, pkg._stream_ptr()), "dump")
    pkg.check(lib.mz_cuda_memcpy_d2d(rows.data_ptr() + 4 * n, len_rows, 4 * n, pkg._stream_ptr()), "dump")
    rows = rows.cpu().numpy().view(np.uint32).astype(np.float64)
    k = DUMP_SAMPLE // world
    pos = np.arange(stream_len) if stream_len <= k else np.sort(np.random.default_rng(0).integers(0, stream_len, k))
    joined = torch.empty(max(stream_len, 1), dtype=torch.uint8, device=dev)
    pkg.check(lib.mz_cuda_memcpy_d2d(joined.data_ptr(), stream, stream_len, pkg._stream_ptr()), "dump")
    sample = joined[torch.from_numpy(pos).to(dev)].cpu().numpy().astype(np.float32)
    del joined
    suffix = "" if world == 1 else "_rank%d" % rank
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("chunk_crc32", rows[:n]), ("chunk_compressed_bytes", rows[n:]),
                      ("totals", np.array([nbytes, stream_len, crc], dtype=np.float64)),
                      ("stream_sample", sample), ("stream_sample_positions", pos.astype(np.float64))):
        np.save(os.path.join(out_dir, name + suffix + ".npy"), arr)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    import textgen
    if args.config != "c5":
        return {"c1": run_c1, "c2": run_c2, "c3": run_c3, "c4": run_c4}[args.config](args, rank, world, local_rank)
    pkg = ge._load_pkg()
    lib = pkg.load()
    torch.cuda.set_device(local_rank)
    pkg.check(lib.mz_cuda_init(), "mz_cuda_init")
    dev = torch.device("cuda", local_rank)
    total = int(args.size_gib * GiB) // 65536 * 65536
    nchunks_total = total // 65536
    c0 = rank * nchunks_total // world
    c1 = (rank + 1) * nchunks_total // world
    shard = (c1 - c0) * 65536
    # ---- input: this rank's shard of the one global buffer (generator is position-independent) -----------------------------
    src = torch.empty(shard, dtype=torch.uint8, device=dev)
    seg = 64 << 20
    for o in range(0, shard, seg):
        k = min(seg, shard - o)
        textgen.device_into(src.data_ptr() + o, k, 1000 + (c0 * 65536 + o) // seg)
    torch.cuda.synchronize()
    # ---- sub-batches: with N>1 the shard is compressed in NB pieces so the all-gather of piece j overlaps the compression of j+1
    NB = 1 if world == 1 else (args.sub_batches if args.sub_batches > 0 else (8 if world >= 8 else 4))  # measured: 4 pieces best at N=2/4, 8 at N=8
    nshard_chunks = c1 - c0
    bounds = [nshard_chunks * j // NB for j in range(NB + 1)]
    subs = [(bounds[j] * 65536, (bounds[j + 1] - bounds[j]) * 65536) for j in range(NB)]  # (byte offset in shard, bytes)
    bounds_chunks = bounds
    batches = [pkg.DeflateBatch(max(nb, 65536)) for _, nb in subs]
    stream = torch.cuda.current_stream()
    comm_stream = torch.cuda.Stream() if world > 1 else None
    ev_done = [torch.cuda.Event() for _ in range(NB)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    # ---- N > 1: the all-gather runs on the COPY ENGINES. Every rank owns one `gathered` buffer (cudaMalloc through the library,
    # exported by IPC handle, mapped by every peer): rank r's joined stream lives at region_off[r] in all of them, its per-chunk
    # {crc32, out_len} rows at chunk index c0 in the global tables. A finished piece is pushed to the N-1 peers with
    # cudaMemcpyAsync on a second stream while the SMs compress the next piece; no SM-based collective competes with the
    # 2 x 111 KB deflate CTAs. Piece offsets come from the warm-up pass: the encoder is bit-reproducible, so they do not change.
    state = {"ready": False, "base": [0] * (NB + 1)}
    if world > 1:
        rbounds = [int(lib.mz_cuda_gather_region_bound(((r + 1) * nchunks_total // world - r * nchunks_total // world) * 65536)) for r in range(world)]
        region_off = [sum(rbounds[:r]) for r in range(world)]
        cap_total = sum(rbounds)
        g_mine = lib.mz_cuda_malloc(cap_total + 256)
        t_crc = lib.mz_cuda_malloc(nchunks_total * 4 + 256)
        t_len = lib.mz_cuda_malloc(nchunks_total * 4 + 256)
        assert g_mine and t_crc and t_len, "cudaMalloc of the gathered buffers failed"
        handles = []
        for ptr in (g_mine, t_crc, t_len):
            h = C.create_string_buffer(64)
            pkg.check(lib.mz_cuda_ipc_export(ptr, h), "ipc_export")
            handles.append(h.raw)
        allh = [None] * world
        dist.all_gather_object(allh, handles)
        peers = []
        for r in range(world):
            if r == rank:
                peers.append((g_mine, t_crc, t_len))
                continue
            got = []
            for hb in allh[r]:
                pp = C.c_void_p()
                pkg.check(lib.mz_cuda_ipc_open(C.create_string_buffer(hb, 64), C.byref(pp)), "ipc_open")
                got.append(pp.value)
            peers.append(tuple(got))
        copy_stream_t = torch.cuda.Stream()
        copy_s = copy_stream_t.cuda_stream
        ev_piece = [lib.mz_cuda_event_create() for _ in range(NB)]

    def compress_sub(j, kev=None):
        off, nb = subs[j]
        b = batches[j]
        n = b.nchunks(nb)
        s = pkg._stream_ptr()
        final = pkg.FLAG_FINAL if (rank == world - 1 and j == NB - 1) else 0  # only the globally last chunk carries BFINAL
        base = src.data_ptr() + off
        if kev is not None:
            kev[0].record(stream)
        pkg.check(lib.mz_cuda_deflate_chunks(base, nb, 65536, None, None, None, n, final, args.level, b.slots.data_ptr(), b.stride,
                                             b.out_len.data_ptr(), s), "deflate")
        if kev is not None:
            kev[1].record(stream)
        cbase = c0 + bounds_chunks[j]  # global index of the piece's first chunk
        crc_dst = b.chunk_crc.data_ptr() if world == 1 else t_crc + 4 * cbase
        pkg.check(lib.mz_cuda_crc32_segments(base, nb, 65536, None, None, n, b.residue.data_ptr(), crc_dst, s), "crc")
        pkg.check(lib.mz_cuda_crc32_fold(b.residue.data_ptr(), n, 65536, nb, b.crc_out.data_ptr(), s), "fold")
        # the join writes straight into this rank's region of its own gathered buffer (N > 1, once the offsets are known)
        dst = b.joined.data_ptr() if not state["ready"] else g_mine + region_off[rank] + state["base"][j]
        pkg.check(lib.mz_cuda_concat(b.slots.data_ptr(), b.stride, b.out_len.data_ptr(), n, b.offsets.data_ptr(), dst, s), "concat")
        return 5

    def step(kevs=None):
        launches = 0
        for j in range(NB):
            launches += compress_sub(j, kevs[j] if kevs else None)
            if world > 1 and state["ready"]:
                off, nb = subs[j]
                n = batches[j].nchunks(nb)
                cbase = c0 + bounds_chunks[j]
                L = state["base"][j + 1] - state["base"][j]
                pkg.check(lib.mz_cuda_memcpy_d2d(t_len + 4 * cbase, batches[j].out_len.data_ptr(), 4 * n, pkg._stream_ptr()), "rows")
                pkg.check(lib.mz_cuda_event_record(ev_piece[j], pkg._stream_ptr()), "event")
                pkg.check(lib.mz_cuda_stream_wait_event(copy_s, ev_piece[j]), "wait")
                for r in range(world):  # THE exchange of the path: piece j of this rank's stream + its rows, to every peer
                    if r == rank:
                        continue
                    pg, pc, pl = peers[r]
                    o = region_off[rank] + state["base"][j]
                    pkg.check(lib.mz_cuda_memcpy_peer(pg + o, g_mine + o, L, copy_s), "peer copy")
                    pkg.check(lib.mz_cuda_memcpy_peer(pc + 4 * cbase, t_crc + 4 * cbase, 4 * n, copy_s), "peer copy")
                    pkg.check(lib.mz_cuda_memcpy_peer(pl + 4 * cbase, t_len + 4 * cbase, 4 * n, copy_s), "peer copy")
        if world > 1 and state["ready"]:
            stream.wait_stream(copy_stream_t)  # the step ends when this rank's pieces have left
        return launches

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def piece_totals():
        return [int(b.offsets[b.nchunks(nb)].item()) for b, (_, nb) in zip(batches, subs)]

    # warm-up: the first pass measures the pieces (their sizes fix where each lands in the gathered buffers), the rest run the full pipeline
    step()
    barrier()
    if world > 1:
        tot = piece_totals()
        for j in range(NB):
            state["base"][j + 1] = state["base"][j] + tot[j]
        assert state["base"][NB] <= rbounds[rank], "region too small"
        state["ready"] = True
    for i in range(max(0, args.warmup - 1) + (1 if world > 1 else 0)):
        step()
    barrier()
    totals = piece_totals()
    comp_bytes = sum(totals)
    clocks = ClockSampler(local_rank)
    clocks.start()
    kev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(NB)] for _ in range(args.steps)]
    barrier()
    ev[0].record(stream)
    launches = 0
    for i in range(args.steps):
        launches += step(kev[i])
    ev[1].record(stream)
    barrier()
    ms = ev[0].elapsed_time(ev[1])
    kms = sum(a.elapsed_time(b) for row in kev for a, b in row) / max(1, args.steps)
    clk = clocks.stop()
    if world > 1:
        assert piece_totals() == [state["base"][j + 1] - state["base"][j] for j in range(NB)], "piece sizes changed between passes"
        # the gathered buffer really holds every rank's stream: the next rank's region must start with a valid block header and its
        # rows must be filled in (spot check), and the rank-ordered concatenation of all regions is checked against the CRC table
        nxt = (rank + 1) % world
        head = torch.empty(16, dtype=torch.uint8, device=dev)
        pkg.check(lib.mz_cuda_memcpy_d2d(head.data_ptr(), g_mine + region_off[nxt], 16, pkg._stream_ptr()), "check")
        nxt_c0 = nxt * nchunks_total // world
        rows = torch.empty(2, dtype=torch.int32, device=dev)
        pkg.check(lib.mz_cuda_memcpy_d2d(rows.data_ptr(), t_len + 4 * nxt_c0, 4, pkg._stream_ptr()), "check")
        torch.cuda.synchronize()
        assert int(head[0].item()) & 6 in (0, 4), "peer region does not start with a stored/dynamic block header"
        assert 0 < int(rows[0].item()) <= 65632, "peer rows missing"
    # CRC of the shard = fold of the pieces' CRCs (host arithmetic); rank 0 reports its own shard's, from the last timed step
    crc_whole = 0
    for j, (b, (_, nb)) in enumerate(zip(batches, subs)):
        c = int(b.crc_out[1].item()) & 0xFFFFFFFF
        crc_whole = c if j == 0 else lib.mz_cuda_crc32_combine(crc_whole, c, nb)
    if args.dump_outputs:
        if world == 1:
            b = batches[0]
            stream, stream_len, crc_rows, len_rows = b.joined.data_ptr(), piece_totals()[0], b.chunk_crc.data_ptr(), b.out_len.data_ptr()
        else:
            stream, stream_len = g_mine + region_off[rank], state["base"][NB]
            crc_rows, len_rows = t_crc + 4 * c0, t_len + 4 * c0
        dump_outputs(args.dump_outputs, rank, world, lib, pkg, dev, shard, crc_whole, stream, stream_len, crc_rows, len_rows)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = (total / GiB) * args.steps / (ms / 1000.0)

    # ---- e2e through the vtbl with host buffers ----------------------------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        import cuharness
        tl = cuharness.TestLib()
        hsrc = torch.empty(shard, dtype=torch.uint8, pin_memory=True)
        hsrc.copy_(src)
        torch.cuda.synchronize()
        sink_cap = shard * 9 // 16 + (64 << 20)  # level-1 text lands near 0.503 of the input; leave room for other data
        hsink = torch.empty(sink_cap, dtype=torch.uint8, pin_memory=True)
        times, times_discard = [], []
        out_bytes = 0
        # the last pass repeats the measurement with a sink that drops the bytes: what is left is upload + kernels + download
        # into the stream's pinned staging, i.e. the codec without the consumer's single-threaded memcpy
        SINK_THREADS = 8
        times_single = []
        for i in range(args.e2e_steps + 3):
            single = i == args.e2e_steps + 1
            discard = i == args.e2e_steps + 2
            sink = tl.lib.mz_stream_mem64_create()
            tl.lib.mz_stream_mem64_set_sink(sink, hsink.data_ptr(), sink_cap)
            tl.lib.mz_stream_mem64_set_copy_threads(sink, 1 if single else SINK_THREADS)
            if discard:
                tl.lib.mz_stream_mem64_set_discard(sink, 1)
            s = lib.mz_stream_cuda_create()
            lib.mz_stream_cuda_set_prop_int64(s, pkg.MZ_STREAM_PROP_COMPRESS_LEVEL, args.level)
            tl.lib.mzt_set_base(s, sink)
            barrier()
            t0 = time.perf_counter()
            assert lib.mz_stream_cuda_open(s, None, pkg.MZ_OPEN_MODE_WRITE) == 0
            wrote = tl.lib.mzt_write_all(s, hsrc.data_ptr(), shard, 1 << 30)
            cerr = lib.mz_stream_cuda_close(s)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            assert wrote == shard and cerr == 0, (wrote, cerr)
            out_bytes = tl.lib.mzt_tell(sink)
            ps = C.c_void_p(s)
            lib.mz_stream_cuda_delete(C.byref(ps))
            tl.delete(sink)
            if discard:
                times_discard.append(dt)
            elif single:
                times_single.append(dt)
            elif i > 0:
                times.append(dt)
            if not discard:
                out_bytes_kept = out_bytes
        out_bytes = out_bytes_kept
        tt = torch.tensor([sum(times) / len(times), times_discard[0], times_single[0]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": round((total / GiB) / float(tt[0].item()), 4), "unit": UNIT, "h2d_bytes_per_step": shard, "d2h_bytes_per_step": int(out_bytes),
               "steps": len(times), "api": "mz_stream_cuda_open/write(1 GiB calls)/close over a 64-bit memory base stream, pinned host input",
               "value_single_thread_sink": round((total / GiB) / float(tt[2].item()), 4),
               "value_discarding_sink": round((total / GiB) / float(tt[1].item()), 4),
               "sink": "host memory stream (tests/support/mem64.c) copying every compressed byte with %d threads" % SINK_THREADS,
               "note": "value_single_thread_sink: the same sink with one memcpy thread (the consumer, not the codec, is then the limit); "
                       "value_discarding_sink: the base stream drops the bytes (upload + kernels + download into pinned staging only)"}
        del hsrc, hsink

    if rank != 0:
        return
    # ---- roofline of the dominant kernel -----------------------------------------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = shard / (kms / 1000.0) / 1e9
    traffic, tsrc = None, None
    for tp in ("r2_deflate_kernel.json", "r1_deflate_kernel.json"):  # the newest committed ncu --set full capture of the kernel
        tp = os.path.join(ROOT, "profiles", tp)
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_input_byte")
                traffic = None if traffic is None else round(traffic * shard / NB)
                tsrc = "profiles/" + os.path.basename(tp)
                break
            except Exception:
                traffic = None
    roofline = {"bound": "hbm", "kernel": "deflate_chunks_kernel", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 5), "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": shard // NB, "ms_per_launch": round(kms / NB, 4), "launches_per_step": NB,
                "traffic_source": "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum per input byte x bytes per launch (%s)" % tsrc}
    cpu = None
    if not args.no_cpu and world == 1:  # reported baseline: rank 0 at N=1 only
        import refshim
        if refshim.ref_available():
            nb = min(args.cpu_sample_mib << 20, shard)
            sample = (C.c_uint8 * nb)()
            arr = src[:nb].cpu().numpy()  # keep the array alive across the copy
            C.memmove(sample, arr.ctypes.data, nb)
            del arr
            cores, cinfo = usable_cores()
            v, thr, comp = cpu_reference_throughput(sample, args.level, threads=cores)
            cpu = {"value": round(v, 4), "unit": UNIT, "cores": thr, "kind": "reference", "host_cores": cinfo,
                   "sample": "first %d MiB of the same buffer, mz_strm_zlib over zlib 1.3 level %d, one independent stream per 4..32 MiB piece on %d host threads "
                             "(affinity capped by the cgroup quota); ratio %.4f" % (nb >> 20, args.level, thr, comp / nb)}
        else:
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "oracle/_ref not built"}
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": workload_text(args),
                   "chunk_bytes": 65536, "level": args.level, "l2": "inputs (%.1f GiB per GPU) are far larger than L2; no flush needed" % (shard / GiB),
                   "parallelism": ("chunk-sharded x%d; per step one all-gather of the bitstreams + per-chunk {crc32, out_len} rows, done with peer-to-peer copies on the copy engines "
                                   "(IPC-mapped gathered buffers, %d pieces per shard overlapped with compression, exact lengths); NCCL only for setup and barriers" % (world, NB)) if world > 1 else "single GPU"},
        "roofline": roofline, "cpu_baseline": cpu, "clocks": clk, "e2e": e2e, "gpu_launches": launches,
        "ratio": round(comp_bytes / shard, 4), "crc32": "%08x" % crc_whole,
    }
    print(json.dumps(line), flush=True)


# ---- the other configurations (BASELINE.json configs[0..3]) -----------------------------------------------------------------
def _peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _setup(local_rank):
    import torch
    import __graft_entry__ as ge
    pkg = ge._load_pkg()
    lib = pkg.load()
    torch.cuda.set_device(local_rank)
    pkg.check(lib.mz_cuda_init(), "mz_cuda_init")
    return torch, pkg, lib, torch.device("cuda", local_rank)


def _emit(args, rank, world, value, ms_per_step, roofline, cpu, clk, e2e, launches, extra=None, l2=None):
    import torch
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms_per_step], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        value = value * ms_per_step / float(t.item())
        ms_per_step = float(t.item())
    if rank != 0:
        return
    metric, unit = METRICS[args.config]
    line = {"metric": metric, "value": round(value, 4), "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak" if world > 1 else "strong", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_text(args), "level": args.level, "l2": l2 or "inputs are larger than L2; no flush needed",
                       "parallelism": "single GPU" if world == 1 else "%d independent replicas (this configuration does not shard)" % world},
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clk, "e2e": e2e, "gpu_launches": launches}
    if extra:
        line.update(extra)
    print(json.dumps(line), flush=True)


def _barrier(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def run_c1(args, rank, world, local_rank):
    """CRC-32 of a 64 MiB buffer (uniform random bytes, seed 1). value: K1 on a device-resident buffer (segments + fold), L2 flushed
    before every timed iteration (64 MiB fits the 126 MB L2); e2e: the replaced symbol mz_crypt_crc32_update on a HOST buffer."""
    torch, pkg, lib, dev = _setup(local_rank)
    import numpy as np
    import zlib
    n = 64 << 20
    host = np.random.default_rng(1).integers(0, 256, n, dtype=np.uint8)
    want = zlib.crc32(host.tobytes())
    src = torch.from_numpy(host).to(dev)
    nseg = n // 65536
    res = torch.empty(nseg, dtype=torch.int32, device=dev)
    out2 = torch.zeros(2, dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    s = pkg._stream_ptr()

    def once():
        pkg.check(lib.mz_cuda_crc32_segments(src.data_ptr(), n, 65536, None, None, nseg, res.data_ptr(), None, s))
        pkg.check(lib.mz_cuda_crc32_fold(res.data_ptr(), nseg, 65536, n, out2.data_ptr(), s))
    for _ in range(max(3, args.warmup)):
        once()
    _barrier(world)
    assert (int(out2[1].item()) & 0xffffffff) == want
    clocks = ClockSampler(local_rank)
    clocks.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b, c in evs:
        flush.fill_(1)  # evict the input from L2 (not timed)
        a.record()
        pkg.check(lib.mz_cuda_crc32_segments(src.data_ptr(), n, 65536, None, None, nseg, res.data_ptr(), None, s))
        b.record()
        pkg.check(lib.mz_cuda_crc32_fold(res.data_ptr(), nseg, 65536, n, out2.data_ptr(), s))
        c.record()
    _barrier(world)
    clk = clocks.stop()
    ms = sum(a.elapsed_time(c) for a, b, c in evs) / args.steps
    kms = sum(a.elapsed_time(b) for a, b, c in evs) / args.steps
    peak, psrc = _peak()
    roofline = {"bound": "hbm", "kernel": "crc32_segments_kernel", "achieved": round(n / kms / 1e6, 2), "peak": peak, "unit": "GB/s",
                "frac": round(n / kms / 1e6 / peak, 5), "traffic": None, "peak_source": psrc, "algorithmic_bytes_per_launch": n,
                "ms_per_launch": round(kms, 5), "launches_per_step": 1}
    # e2e: the drop-in symbol with host memory (pageable, as the reference's callers have it; and pinned)
    hb = C.create_string_buffer(host.tobytes(), n)
    times, times_pin = [], []
    hp = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    hp.copy_(torch.from_numpy(host))
    for i in range(args.e2e_steps + 2):
        t0 = time.perf_counter()
        got = lib.mz_crypt_crc32_update(0, hb, n)
        dt = time.perf_counter() - t0
        assert got == want
        t0 = time.perf_counter()
        got = lib.mz_crypt_crc32_update(0, C.c_void_p(hp.data_ptr()), n)
        dtp = time.perf_counter() - t0
        assert got == want
        if i >= 2:
            times.append(dt)
            times_pin.append(dtp)
    e2e = {"value": round(n / GiB / (sum(times) / len(times)), 4), "unit": "GiB/s", "h2d_bytes_per_step": n, "d2h_bytes_per_step": 8,
           "api": "mz_crypt_crc32_update(0, host buffer, 64 MiB): pageable caller memory, copied through pinned staging in 8 MiB pieces",
           "value_pinned_caller": round(n / GiB / (sum(times_pin) / len(times_pin)), 4)}
    cpu = None
    if not args.no_cpu and world == 1:
        import refshim
        if refshim.ref_available():
            ref = refshim.RefLib()
            ts = []
            for i in range(4):
                t0 = time.perf_counter()
                ref.lib.mz_crypt_crc32_update(0, host.ctypes.data, n)
                ts.append(time.perf_counter() - t0)
            cpu = {"value": round(n / GiB / min(ts[1:]), 4), "unit": "GiB/s", "cores": 1, "kind": "reference",
                   "sample": "the same 64 MiB through the reference's mz_crypt_crc32_update (zlib 1.3 crc32), one core (the call is single-threaded)"}
    _emit(args, rank, world, n / GiB / (ms / 1000.0), ms, roofline, cpu, clk, e2e, 2 * args.steps, {"crc32": "%08x" % want},
          l2="64 MiB fits L2: a 256 MiB buffer is rewritten before every timed iteration")


def run_c2(args, rank, world, local_rank):
    """minigzip-style: DEFLATE level 6 with gzip framing of 256 MiB text. value: K2+K3 + K1 + K4 on the device-resident buffer;
    e2e: mz_stream_cuda_open/write/close with window bits 31 and host buffers, checked by CPython zlib."""
    torch, pkg, lib, dev = _setup(local_rank)
    import textgen
    import zlib
    import cuharness
    n = int(args.size_gib * GiB) // 65536 * 65536
    src = textgen.device(n, seed=1234)
    b = pkg.DeflateBatch(n)
    s = pkg._stream_ptr()
    stream = torch.cuda.current_stream()
    nch = b.nchunks(n)

    def step(ev=None):
        if ev:
            ev[0].record(stream)
        pkg.check(lib.mz_cuda_deflate_chunks(src.data_ptr(), n, 65536, None, None, None, nch, pkg.FLAG_FINAL | pkg.FLAG_DICT, args.level, b.slots.data_ptr(), b.stride,
                                             b.out_len.data_ptr(), s), "deflate")
        if ev:
            ev[1].record(stream)
        pkg.check(lib.mz_cuda_crc32_segments(src.data_ptr(), n, 65536, None, None, nch, b.residue.data_ptr(), b.chunk_crc.data_ptr(), s), "crc")
        pkg.check(lib.mz_cuda_crc32_fold(b.residue.data_ptr(), nch, 65536, n, b.crc_out.data_ptr(), s), "fold")
        pkg.check(lib.mz_cuda_concat(b.slots.data_ptr(), b.stride, b.out_len.data_ptr(), nch, b.offsets.data_ptr(), b.joined.data_ptr(), s), "concat")
    for _ in range(max(3, args.warmup)):
        step()
    _barrier(world)
    comp = int(b.offsets[nch].item())
    clocks = ClockSampler(local_rank)
    clocks.start()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _barrier(world)
    e0.record(stream)
    for i in range(args.steps):
        step(kev[i])
    e1.record(stream)
    _barrier(world)
    clk = clocks.stop()
    ms = e0.elapsed_time(e1) / args.steps
    kms = sum(a.elapsed_time(c) for a, c in kev) / args.steps
    peak, psrc = _peak()
    roofline = {"bound": "hbm", "kernel": "deflate_chunks_kernel", "achieved": round(n / kms / 1e6, 2), "peak": peak, "unit": "GB/s",
                "frac": round(n / kms / 1e6 / peak, 5), "traffic": None, "peak_source": psrc, "algorithmic_bytes_per_launch": n,
                "ms_per_launch": round(kms, 4), "launches_per_step": 1}
    e2e = None
    if not args.no_e2e:
        tl = cuharness.TestLib()
        hsrc = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        hsrc.copy_(src)
        torch.cuda.synchronize()
        cap = n * 9 // 16 + (64 << 20)
        hsink = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
        times = []
        for i in range(args.e2e_steps + 1):
            sink = tl.lib.mz_stream_mem64_create()
            tl.lib.mz_stream_mem64_set_sink(sink, hsink.data_ptr(), cap)
            z = lib.mz_stream_cuda_create()
            lib.mz_stream_cuda_set_prop_int64(z, pkg.MZ_STREAM_PROP_COMPRESS_LEVEL, args.level)
            lib.mz_stream_cuda_set_prop_int64(z, pkg.MZ_STREAM_PROP_COMPRESS_WINDOW, 31)
            tl.lib.mzt_set_base(z, sink)
            t0 = time.perf_counter()
            assert lib.mz_stream_cuda_open(z, None, pkg.MZ_OPEN_MODE_WRITE) == 0
            wrote = tl.lib.mzt_write_all(z, hsrc.data_ptr(), n, 1 << 20)  # 1 MiB writes; minigzip itself uses 16 KiB ones
            cerr = lib.mz_stream_cuda_close(z)
            dt = time.perf_counter() - t0
            assert wrote == n and cerr == 0
            out_bytes = tl.lib.mzt_tell(sink)
            pz = C.c_void_p(z)
            lib.mz_stream_cuda_delete(C.byref(pz))
            tl.delete(sink)
            if i > 0:
                times.append(dt)
        gz = bytes(hsink[:out_bytes].numpy().tobytes())
        back = zlib.decompress(gz, 31)
        assert len(back) == n and zlib.crc32(back) == zlib.crc32(hsrc.numpy().tobytes()), "gzip written through the vtbl does not round-trip"
        e2e = {"value": round(n / GiB / (sum(times) / len(times)), 4), "unit": "GiB/s", "h2d_bytes_per_step": n, "d2h_bytes_per_step": int(out_bytes),
               "api": "mz_stream_cuda_open/write(1 MiB calls)/close, window bits 31 (gzip), pinned host input, host memory sink; output checked by CPython zlib",
               "ratio": round(out_bytes / n, 4)}
    cpu = None
    if not args.no_cpu and world == 1:
        import refshim
        if refshim.ref_available():
            nb = min(n, 64 << 20)
            sample = (C.c_uint8 * nb)()
            arr = src[:nb].cpu().numpy()
            C.memmove(sample, arr.ctypes.data, nb)
            v1, _, comp1 = cpu_reference_throughput(sample, args.level, threads=1, window_bits=31, piece=nb)
            cpu = {"value": round(v1, 4), "unit": "GiB/s", "cores": 1, "kind": "reference",
                   "sample": "first %d MiB of the same buffer through ONE mz_stream_zlib (level %d, gzip) on one core -- minigzip is single-threaded; ratio %.4f" % (nb >> 20, args.level, comp1 / nb)}
    _emit(args, rank, world, n / GiB / (ms / 1000.0), ms, roofline, cpu, clk, e2e, 4 * args.steps, {"ratio": round(comp / n, 4)})


def run_c3(args, rank, world, local_rank):
    """One multi-block gzip member (zlib level 6 blocks, see make_gzip_member) of size-gib GiB of text, read through
    mz_stream_cuda_read with host buffers (1 MiB reads): CRC, ISIZE (mod 2^32) and TOTAL_IN checked. The read path has no
    device-resident variant (the caller's buffer is host memory by contract), so value == e2e."""
    torch, pkg, lib, dev = _setup(local_rank)
    import textgen
    import zlib
    import cuharness
    tl = cuharness.TestLib()
    n = int(args.size_gib * GiB)
    text = textgen.host_buffer(n, seed=4321)
    member, crc = make_gzip_member(text, n, 6)
    del text
    msrc = C.create_string_buffer(member, len(member))
    clen = len(member)
    del member
    out = torch.empty(n + 4096, dtype=torch.uint8, pin_memory=False)
    out.fill_(1)  # touch the pages outside the timed region
    times = []
    clocks = ClockSampler(local_rank)
    trace = None
    for i in range(min(args.warmup, 1) + min(args.steps, 3) + 1):
        last = i == min(args.warmup, 1) + min(args.steps, 3)
        if last:  # one extra, untimed pass with per-kernel times on stderr (serialises the rounds)
            os.environ["MZ_CUDA_TRACE"] = "1"
            tf = tempfile.TemporaryFile()
            saved = os.dup(2)
            os.dup2(tf.fileno(), 2)
        if i == min(args.warmup, 1):
            clocks.start()
        srcs = tl.lib.mz_stream_mem64_create()
        tl.lib.mz_stream_mem64_set_buffer(srcs, msrc, clen)
        z = lib.mz_stream_cuda_create()
        tl.lib.mzt_set_prop(z, pkg.MZ_STREAM_PROP_COMPRESS_WINDOW, 31)
        tl.lib.mzt_set_base(z, srcs)
        t0 = time.perf_counter()
        assert tl.lib.mzt_open(z, None, pkg.MZ_OPEN_MODE_READ) == 0
        got = tl.lib.mzt_read_all(z, out.data_ptr(), n + 1024, 1 << 20)
        cerr = tl.lib.mzt_close(z)
        dt = time.perf_counter() - t0
        tin = tl.get_prop(z, pkg.MZ_STREAM_PROP_TOTAL_IN)[1]
        tl.delete(z)
        tl.delete(srcs)
        if last:
            os.dup2(saved, 2)
            os.close(saved)
            tf.seek(0)
            trace = tf.read().decode(errors="replace")
            os.environ.pop("MZ_CUDA_TRACE", None)
        assert got == n and cerr == 0 and tin == clen, (got, cerr, tin, clen)
        if i >= min(args.warmup, 1) and not last:
            times.append(dt)
    clk = clocks.stop()
    crc_out = zlib.crc32(memoryview(out.numpy())[:n])
    assert crc_out == crc, "output CRC differs from the member's"
    sec = sum(times) / len(times)
    # dominant kernels from the trace: sums over the rounds of the pass
    ksum = {"find": 0.0, "scan": 0.0, "chain": 0.0, "resolve": 0.0, "emit": 0.0}
    rounds = 0
    import re
    for m in re.finditer(r"K6 kernels ms: find ([\d.]+) scan ([\d.]+) chain ([\d.]+) compose\+link\+resolve ([\d.]+) emit ([\d.]+)", trace or ""):
        rounds += 1
        for k, v in zip(("find", "scan", "chain", "resolve", "emit"), m.groups()):
            ksum[k] += float(v)
    peak, psrc = _peak()
    dom = max(("scan", "emit"), key=lambda k: ksum[k])
    kms = ksum[dom] or sec * 1000
    roofline = {"bound": "hbm", "kernel": "inflate_spec_%s_kernel" % dom, "achieved": round((n + clen) / kms / 1e6, 2), "peak": peak, "unit": "GB/s",
                "frac": round((n + clen) / kms / 1e6 / peak, 5), "traffic": None, "peak_source": psrc,
                "algorithmic_bytes_per_launch": (n + clen) // max(rounds, 1), "ms_per_launch": round(kms / max(rounds, 1), 4), "launches_per_step": rounds,
                "kernel_ms_per_step": {k: round(v, 2) for k, v in ksum.items()},
                "note": "algorithmic bytes = output written + compressed read; kernel times from one extra pass with MZ_CUDA_TRACE=1 (serialised rounds)"}
    e2e = {"value": round(n / GiB / sec, 4), "unit": "GiB/s", "h2d_bytes_per_step": clen, "d2h_bytes_per_step": n,
           "api": "mz_stream_cuda_open/read(1 MiB calls)/close over a 64-bit memory base stream, window bits 31, pageable host output"}
    cpu = None
    if not args.no_cpu and world == 1:
        import refshim
        if refshim.ref_available():
            ref = refshim.RefLib()
            nb = 256 << 20
            t2 = textgen.host_buffer(nb, seed=4321)
            m2, _ = make_gzip_member(t2, nb, 6)
            t0 = time.perf_counter()
            o2 = ref.zlib_decompress(m2, window_bits=31, read_size=1 << 16)
            dt = time.perf_counter() - t0
            assert len(o2) == nb
            cpu = {"value": round(nb / GiB / dt, 4), "unit": "GiB/s", "cores": 1, "kind": "reference",
                   "sample": "a 256 MiB member of the same text through mz_stream_zlib_read (64 KiB reads), one core: one member cannot be split across cores"}
    _emit(args, rank, world, n / GiB / sec, sec * 1000, roofline, cpu, clk, e2e, rounds * 7, {"ratio": round(clen / n, 4), "crc32": "%08x" % crc, "isize_mod32": n & 0xffffffff})


def run_c4(args, rank, world, local_rank):
    """zip of N x 64 KiB entries (70 % text, 20 % records, 10 % incompressible), level 6, archive on tmpfs, driven by the C program
    oracle/_ref/zipbatch_cuda (tests/support/zipbatch.c). The product's native archive writer (mz_zip_cuda_write_archive: headers,
    streams, central directory by the library, a round's region assembled on the device) is the measured path; the batch writer on
    the reference's raw-entry seam (mz_zip_cuda_add_buffers) is reported beside it. With N GPUs the ENTRIES shard across the GPUs
    inside one writer (rounds go round-robin to the devices, flag MZ_ZIP_CUDA_ALL_DEVICES): a zip archive is one serial byte
    stream, so rank 0 drives all N devices from one process and the other ranks only take part in the barriers."""
    torch, pkg, lib, dev = _setup(local_rank)
    exe = os.path.join(ROOT, "oracle", "_ref", "zipbatch_cuda")
    entries = int(round(args.size_gib * GiB / 65536))
    runs, seam = [], None
    clocks = ClockSampler(local_rank)
    clk = None
    if rank == 0:
        d = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        env = dict(os.environ)  # under torchrun every rank sees all devices: the writer takes them all
        mode = "native_all" if world > 1 else "native"
        try:
            # ONE writer process writes the archive warm-up + steps times (ZIPBATCH_REPEAT): like the other configs' warm-up steps, the
            # timed ones run in a warm process -- CUDA context up, the library's staging pool filled by the first archive
            nw, ns = min(args.warmup, 1), min(args.steps, 3)
            env["ZIPBATCH_REPEAT"] = str(nw + ns)
            clocks.start()
            r = subprocess.run([exe, os.path.join(d, "c4.zip"), str(entries), "65536", str(args.level), mode], stdout=subprocess.PIPE, text=True, env=env, timeout=1800)
            lines = [json.loads(x) for x in r.stdout.strip().splitlines() if x.startswith("{")]
            assert len(lines) == nw + ns and all(j["err"] == 0 and j["close_err"] == 0 for j in lines), r.stdout[-2000:]
            first_archive = lines[0]
            runs = lines[nw:]
            env.pop("ZIPBATCH_REPEAT")
            clk = clocks.stop()
            import zipfile
            with zipfile.ZipFile(os.path.join(d, "c4.zip")) as zf:  # a valid zip: CPython's zipfile checks every entry's CRC
                assert len(zf.namelist()) == entries and zf.testzip() is None
            if world == 1:
                r = subprocess.run([exe, os.path.join(d, "c4s.zip"), str(entries), "65536", str(args.level), "cuda"], stdout=subprocess.PIPE, text=True, env=env, timeout=900)
                seam = json.loads(r.stdout.strip().splitlines()[-1])
        finally:
            subprocess.run(["rm", "-rf", d])
    _barrier(world)
    if rank != 0:
        return
    add_s = sum(j["add_s"] + j["close_s"] for j in runs) / len(runs)
    gpu_ms = sum(j["gpu_ms"] for j in runs) / len(runs)
    nbytes = runs[-1]["bytes_in"]
    peak, psrc = _peak()
    roofline = {"bound": "hbm", "kernel": "deflate_chunks_kernel (+ crc32_segments, gather, header scatter)", "achieved": round(nbytes / gpu_ms / 1e6, 2), "peak": peak,
                "unit": "GB/s", "frac": round(nbytes / gpu_ms / 1e6 / peak, 5), "traffic": None, "peak_source": psrc,
                "algorithmic_bytes_per_launch": nbytes // max(runs[-1]["rounds"], 1), "ms_per_launch": round(gpu_ms / max(runs[-1]["rounds"], 1), 3),
                "launches_per_step": runs[-1]["rounds"],
                "note": "gpu_ms = per round: kernels + table download + layout + region assembly + region download, host clock of the worker thread (summed over devices)"}
    value = nbytes / GiB / add_s
    e2e = {"value": round(value, 4), "unit": "GiB/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": runs[-1]["bytes_out"],
           "api": "mz_zip_cuda_write_archive(file stream, %d host buffers, flags %s), archive file on tmpfs" % (entries, "ALL_DEVICES" if world > 1 else "0"),
           "entries_per_s": round(entries / add_s, 1), "pack_ms": runs[-1]["pack_ms"], "gpu_ms": runs[-1]["gpu_ms"], "write_ms": runs[-1]["container_ms"],
           "setup_ms": runs[-1].get("setup_ms"), "cuda_init_s_not_in_the_timed_region": runs[-1].get("cuda_init_s"),
           "first_archive_of_the_process": {"entries_per_s": first_archive["entries_per_s"], "setup_ms": first_archive.get("setup_ms")},
           "note": "timed: the whole mz_zip_cuda_write_archive call (staging from the library's pool, rounds, central directory, release) + close of the "
                   "file stream, in a process that has written the archive once before (warm-up step: CUDA context, page-locked staging pool); the "
                   "first archive of the process is reported beside it; pack_ms is summed over the four round workers"}
    if seam:
        e2e["raw_entry_seam"] = {"entries_per_s": seam["entries_per_s"], "GiB_per_s": seam["GiB_per_s"], "container_ms": seam["container_ms"],
                                 "api": "mz_zip_cuda_add_buffers: the reference's container writes every header (three calls per entry)"}
    cpu = None
    if not args.no_cpu and world == 1:
        ref_exe = os.path.join(ROOT, "oracle", "_ref", "zipbatch_ref")
        if os.path.exists(ref_exe):
            d2 = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
            try:
                r = subprocess.run([ref_exe, os.path.join(d2, "r.zip"), "6000", "65536", str(args.level), "ref"], stdout=subprocess.PIPE, text=True, timeout=600)
                j = json.loads(r.stdout.strip().splitlines()[-1])
                cpu = {"value": j["GiB_per_s"], "unit": "GiB/s", "cores": 1, "kind": "reference", "entries_per_s": j["entries_per_s"],
                       "sample": "6000 entries x 64 KiB through the reference's zip writer (mz_zip_entry_write_open raw=0, zlib level %d, CRC per 64 KiB), one core" % args.level}
            finally:
                subprocess.run(["rm", "-rf", d2])
    metric, unit = METRICS[args.config]
    line = {"metric": metric, "value": round(value, 4), "unit": unit, "n_gpus": world, "steps": len(runs), "warmup": min(args.warmup, 1),
            "ms_per_step": round(add_s * 1000, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_text(args), "level": args.level, "l2": "inputs are larger than L2; no flush needed",
                       "parallelism": "single GPU" if world == 1 else "entries sharded over %d GPUs inside one archive writer (rounds round-robin); one process drives all devices" % world},
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clk, "e2e": e2e, "gpu_launches": 5 * runs[-1]["rounds"],
            "entries": entries, "entries_per_s": round(entries / add_s, 1), "ratio": round(runs[-1]["bytes_out"] / nbytes, 4)}
    print(json.dumps(line), flush=True)


def main():
    faulthandler.enable()
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
