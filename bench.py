#!/usr/bin/env python
"""bench.py — the `deft4j optimise -m NONE` hot path on B200 (BASELINE.json metric: input MB/s optimised).

A step = one pass of the whole path (parse -> optimise -> write -> checksums) over one batch of synthetic input.

  value  : whole-job MB/s of input deflate with the inputs already resident in HBM (deft4cu_device_batch_run)
  e2e    : the same through the reference-facing batch entry of the C ABI (deft4cu_optimise_batch) with pinned HOST
           buffers in and host buffers out, host<->device copies inside the timed region
  roofline / cpu_baseline : see DESIGN.md "Measurement"
  output_verified : after the timed loops the rewritten streams of the last step are inflated with zlib and compared
           (length, CRC-32, Adler-32) with the inflate of the input and with the checksums the device computed
  shapes : short runs of the other named shapes (C3 PNG IDAT batch, C4 ZIP entry mix, C5 adversarial, and the very
           sample the CPU reference arm is timed on), sharded by stream over the ranks (strong scaling over one list)
  per_rank : every rank's own step time and kernel-family times (N > 1)

Launch: `python bench.py --gpus N --steps K --warmup W` (N=1) or under torch.distributed.run with N ranks (one
process per GPU; C2's single stream is replicated per rank, stream lists are sharded by rank: no data-path collective,
the process group is gloo and only carries barriers, timings and result lists).
`--impl reference` times the CPU restatement of the reference (oracle/, the reference itself is Java and this image
has no JVM) with every host core on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step computed as .npy files (dump_outputs).  The inputs come from fixed
seeds, so two builds run with the same arguments can be compared output for output (`--workload ref` also sizes its
sample by the host's core count).
"""
import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the tree may be read-only: the benchmark writes nothing into it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "input MB/s optimised (-m NONE)"
C2_WHY_NO_MERGE = ("--no-merge-blocks: on stationary text every adjacent merge saves a header, so mergeBlocks() "
                   "(DeflateStream.java:568-650) cascades the whole stream into ONE block, re-running optimiseBlock on the "
                   "growing union each time (quadratic; the oracle turns 29 blocks into 1 at 660 KB and needs 4.5x the "
                   "time) - not computable at 1 GiB by any implementation of these semantics, the reference included, "
                   "which is why its own runTestOpt.sh:10-11 uses this flag for its large fixtures; merge-on throughput "
                   "is reported per shape under `shapes`")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4", "c5", "ref"])
    ap.add_argument("--size-mib", type=float, default=float(os.environ.get("DEFT4CU_BENCH_MIB", "1024")),
                    help="C2: size of the single raw deflate stream per GPU (BASELINE config: 1024)")
    ap.add_argument("--count", type=int, default=0, help="C3/C4: streams per GPU (default 12500 / 1250)")
    ap.add_argument("--merge", type=int, default=-1, help="mergeBlocks; default: 0 for C2 (see DESIGN.md), 1 otherwise")
    ap.add_argument("--sample-seconds", type=float, default=30.0, help="CPU baseline budget per sample")
    ap.add_argument("--no-shapes", action="store_true", help="skip the short C3/C4/C5 runs")
    ap.add_argument("--no-verify", action="store_true", help="skip inflating the output of the last timed step")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


def workload_config(a):
    merge = a.merge if a.merge >= 0 else (0 if a.workload == "c2" else 1)
    if a.workload == "c2":
        name = ("single %d MiB raw deflate stream per GPU, zlib level 6 dynamic blocks over synthetic Zipf text "
                "(BASELINE configs[1]), %s" % (a.size_mib, "merge blocks" if merge else "--no-merge-blocks"))
    elif a.workload == "c3":
        a.count = a.count or 12500
        name = "%d synthetic 256x256 RGBA PNG IDAT streams per GPU (BASELINE configs[2]), merge blocks" % a.count
    elif a.workload == "c4":
        a.count = a.count or 1250
        name = "%d ZIP-entry deflate payloads per GPU mixing stored/fixed/dynamic (BASELINE configs[3]), merge blocks" % a.count
    elif a.workload == "c5":
        name = "adversarial streams (BASELINE configs[4]): len-258 / dist-1 and dist-32768 matches at 8 MiB, RLE-heavy headers"
    else:
        name = "the CPU reference arm's own sample (C2-style streams, one or two per host core)"
    return name, merge


def make_streams(a, rank):
    import workloads as W
    if a.workload == "c2":
        # every rank optimises the SAME stream (replicas): per-rank times are then comparable
        return [W.c2_stream(int(a.size_mib * (1 << 20)), seed=0xDEF7)]
    if a.workload == "c3":
        return W.c3_streams(a.count, first=rank * a.count)
    if a.workload == "c4":
        return W.c4_streams(a.count, seed=4 + rank)
    if a.workload == "c5":
        return W.c5_streams(scale=8)
    return reference_sample("c2", os.cpu_count() or 1, a.sample_seconds)[0]


# ---- CPU baseline: the oracle on every host core, one process per stream -------------------------------------------
def _oracle_job(args):
    raw, merge = args
    import oracle_lib
    s = oracle_lib.OracleDeflateStream()
    assert s.parse(raw)
    t0 = time.perf_counter()
    s.optimise(bool(merge))
    s.asBytes()
    return time.perf_counter() - t0


def _oracle_out(args):
    """(saved bits, output bytes, consumed, crc32, adler32, uncompressed length) of the oracle for one stream: the
    checker used by the parity tests."""
    raw, merge = args
    import oracle_lib
    s = oracle_lib.OracleDeflateStream()
    assert s.parse(raw)
    saved = s.optimise(bool(merge))
    out = s.asBytes()
    crc, adler, n = s.getChecksums()
    return saved, out, s.consumed, crc, adler, n


ORACLE_KBPS_PER_CORE = 45e3   # C2 input bytes per second of one oracle thread (no merge), measured on this pool's hosts


def reference_sample(workload, cores, seconds):
    """THE bounded sample both CPU legs use (`cpu_baseline` inside our arm and `--impl reference`): deterministic
    streams of the workload's kind, two per host core, sized so that all cores together need about `seconds`."""
    import workloads as W
    if workload in ("c2", "ref"):
        text_bytes = int(ORACLE_KBPS_PER_CORE * 2.4 * seconds / 2)
        out = []
        for k in range(2 * cores):
            co = zlib.compressobj(6, zlib.DEFLATED, -15, 8)
            out.append(co.compress(W.c2_text(text_bytes, seed=0xBA5E + k)) + co.flush())
        return out, "%d independent C2-style streams of %d KiB text each (two per core)" % (2 * cores, text_bytes >> 10)
    if workload == "c3":
        n = max(cores, int(cores * seconds / 1.5))
        return W.c3_streams(n, first=5_000_000), "%d C3 PNG IDAT streams" % n
    if workload == "c4":
        n = max(cores, int(cores * seconds / 0.8))
        return W.c4_streams(n, seed=99), "%d C4 entry payloads" % n
    return W.c5_streams(scale=1), "the C5 adversarial streams at 1 MiB"


def jvm_probe():
    """The reference is Java: say whether this box could have run it (it cannot be built without /root/reference,
    which only exists in the build container, and that container has no JDK: DESIGN.md 'Oracle')."""
    j, jc = shutil.which("java"), shutil.which("javac")
    return "java=%s javac=%s" % (j or "absent", jc or "absent")


def run_cpu_baseline(a, merge, budget_s, streams=None, what=None):
    import oracle_lib
    oracle_lib.build()
    cores = os.cpu_count() or 1
    if streams is None:
        streams, what = reference_sample(a.workload, cores, budget_s)
    t0 = time.perf_counter()
    with mp.get_context("spawn").Pool(cores) as pool:
        pool.map(_oracle_job, [(s, merge) for s in streams], chunksize=1)
    dt = time.perf_counter() - t0
    total = sum(len(s) for s in streams)
    return {"value": total / dt / 1e6, "unit": "MB/s", "cores": cores, "kind": "port",
            "value_per_core": total / dt / 1e6 / cores, "merge_blocks": bool(merge), "seconds": dt, "jvm": jvm_probe(),
            "sample": "%s, %.2f MB of input deflate in %.1f s; the reference is Java (no JVM in this image), so this is "
                      "the C++ restatement (oracle/), which is faster than the JVM original" % (what, total / 1e6, dt)}


# ---- clocks -------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.

    In-process NVML (nvidia_ml_py) on a thread: a spawned `nvidia-smi -lms` holds up the host side of CUDA calls in every
    process of the box for 0.1-0.5 s at start-up and again at every sample on a multi-GPU box, which starves a GPU that
    runs short kernels (measured: C3 on 2 GPUs 507 instead of 110 ms per step).  NVML is initialised before the warm-up
    steps; only samples taken after mark() count.  Falls back to `nvidia-smi` when the module is missing."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device, period=0.1):
        import threading
        self.samples = []          # (time, sm MHz, max MHz, reasons bitmask)
        self.t_mark = 0.0
        self.p = self.f = None
        self.nv = None
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES renumbers CUDA devices, NVML does not: go through the PCI bus id
            try:
                import torch
                bus = getattr(torch.cuda.get_device_properties(device), "pci_bus_id", None)
            except Exception:  # noqa: BLE001
                bus = None
            h = None
            if bus is not None:
                for k in range(pynvml.nvmlDeviceGetCount()):
                    hk = pynvml.nvmlDeviceGetHandleByIndex(k)
                    if pynvml.nvmlDeviceGetPciInfo(hk).bus == bus:
                        h = hk
                        break
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.nv, self.h = pynvml, h
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def loop():
                while not self._stop.is_set():
                    try:
                        mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        rs = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                        self.samples.append((time.time(), mhz, rs))
                    except Exception:  # noqa: BLE001
                        pass
                    self._stop.wait(period)

            self.th = threading.Thread(target=loop, daemon=True)
            self.th.start()
            return
        except Exception:  # noqa: BLE001 - no NVML module: the command-line tool
            self.nv = None
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "500"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def wait_ready(self, timeout=5.0):
        """the first sample is there: start-up is over"""
        t0 = time.time()
        while time.time() - t0 < timeout:
            if self.nv is not None:
                if self.samples:
                    return
            elif self.p is None or self.p.poll() is not None or os.path.getsize(self.f.name) > 0:
                return
            time.sleep(0.02)

    def mark(self):
        self.t_mark = time.time()

    def stop(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        if self.nv is not None:
            nv = self.nv
            self._stop.set()
            self.th.join(timeout=2)
            bits = [nv.nvmlClocksEventReasonHwSlowdown, nv.nvmlClocksEventReasonHwThermalSlowdown,
                    nv.nvmlClocksEventReasonSwThermalSlowdown, nv.nvmlClocksEventReasonSwPowerCap]
            inside = [x for x in self.samples if x[0] >= self.t_mark - 0.05] or self.samples[-1:]
            reasons = sorted({n for _, _, rs in inside for n, b in zip(names, bits) if rs & b})
            sm = [x[1] for x in inside]
            try:
                nv.nvmlShutdown()
            except Exception:  # noqa: BLE001
                pass
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        import datetime
        for line in self.f:
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if ts < self.t_mark - 0.1:
                    continue
            except ValueError:
                pass
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.f.name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


FAMILIES = ["parse_count", "emit", "lz77", "optimise", "finish_merge", "write", "checksums", "parse_rewalks"]


# ---- the reference arm -----------------------------------------------------------------------------------------------
def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name, merge = workload_config(a)
    cores = os.cpu_count() or 1
    streams, what = reference_sample(a.workload, cores, a.sample_seconds)
    vals, base = [], None
    # one warm-up sample pages the library in; every timed step is the same bounded sample
    for i in range(min(a.warmup, 1) + a.steps):
        base = run_cpu_baseline(a, merge, a.sample_seconds, streams, what)
        if i >= min(a.warmup, 1):
            vals.append(base["value"])
    v = sum(vals) / len(vals)
    base["value"] = v
    base["value_per_core"] = v / cores
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "MB/s", "n_gpus": a.gpus, "steps": a.steps,
                      "warmup": a.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "u8", "data": "synthetic", "config": {"workload": name, "merge_blocks": bool(merge)},
                      "cpu_baseline": base,
                      "e2e": {"value": v, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ---- our arm ---------------------------------------------------------------------------------------------------------
class Ctx:
    """Process-group plumbing: gloo only (barriers, timings, result lists): the data path has no collective."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
        torch.cuda.set_device(self.local)
        os.environ["DEFT4CU_DEVICE"] = str(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("gloo")
            self.dist = dist

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist:
            self.dist.barrier()

    def gather(self, obj):
        if not self.dist:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def max(self, x):
        return max(self.gather(x))

    def sum(self, x):
        return sum(self.gather(x))


def measure(ctx, L, N, streams, merge, steps, warmup, sample_clocks=False, verify=False, e2e_steps=None, dump=None):
    """value (device-resident, CUDA events on the launching stream), e2e (pinned host buffers through the batch
    entry), kernel-family times, launches, output verification — for this rank's `streams`.  With `dump`, the results
    of the last timed step are written there (dump_outputs)."""
    torch = ctx.torch
    n = len(streams)
    in_bytes = sum(len(s) for s in streams)
    out = {"n": n, "in_bytes": in_bytes}
    ptrs, lens = N.make_ptr_arrays(streams)
    stream = torch.cuda.Stream()
    fam = [0.0] * 8
    launches = C.c_uint64(0)
    h = C.c_void_p()
    if n:
        rc = L.deft4cu_device_batch_create(ptrs, lens, n, C.byref(h))
        assert rc == 0, N.last_error()

    def step():
        if not n:
            return
        rc = L.deft4cu_device_batch_run(h, merge, C.byref(launches), C.c_void_p(stream.cuda_stream))
        assert rc == 0, N.last_error()

    with torch.cuda.stream(stream):
        sampler = ClockSampler(ctx.local) if sample_clocks and ctx.rank == 0 else None
        if sampler:
            sampler.wait_ready()
        ctx.barrier()
        for _ in range(warmup):
            step()
        ctx.barrier()
        if sampler:
            sampler.mark()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        total_launches = 0
        for _ in range(steps):
            step()
            total_launches += launches.value
            if n:
                ms = (C.c_float * 8)()
                L.deft4cu_device_batch_timings(h, ms, 8)
                fam = [x + y for x, y in zip(fam, ms)]
        ev1.record(stream)
        ctx.barrier()
        out["clocks"] = sampler.stop() if sampler else None
    out["dev_ms"] = ev0.elapsed_time(ev1)
    out["launches"] = total_launches
    out["fam"] = [x / max(1, steps) for x in fam]
    out["out_bytes"] = out["unc_bytes"] = out["saved_bits"] = 0
    out["verified"] = None
    if n:
        res = (N.Result * n)()
        assert L.deft4cu_device_batch_fetch(h, res) == 0, N.last_error()
        assert all(r.status == 0 for r in res), [r.status for r in res if r.status]
        out["out_bytes"] = sum(r.out_len for r in res)
        out["unc_bytes"] = sum(r.uncompressed_len for r in res)
        out["saved_bits"] = sum(r.saved_bits for r in res)
        if dump:
            dump_outputs(dump, N, res)
        if verify:
            t0 = time.time()
            drift = 0
            for raw, r in zip(streams, res):
                drift += abs(verify_stream(raw, C.string_at(r.out, r.out_len), r))
            out["verified"] = {"streams": n, "seconds": round(time.time() - t0, 1), "abs_bits_size_delta_minus_saved": drift}
        L.deft4cu_free_results(res, n)
        L.deft4cu_device_batch_free(h)
    # ---- e2e: pinned host buffers through the batch entry of the C ABI -----------------------------------------------
    e2e_steps = e2e_steps or steps
    out["e2e_s"] = 0.0
    out["d2h"] = 0
    if n:
        pinned = [torch.frombuffer(bytearray(s), dtype=torch.uint8).pin_memory() for s in streams]
        pp = (C.c_char_p * n)(*[C.cast(t.data_ptr(), C.c_char_p) for t in pinned])
        e2e_res = (N.Result * n)()
        if warmup > 0:  # one untimed call: the library pins its result block on first use
            rc = L.deft4cu_optimise_batch(pp, lens, n, merge, e2e_res)
            assert rc == 0, N.last_error()
            L.deft4cu_free_results(e2e_res, n)
    ctx.barrier()
    t0 = time.perf_counter()
    if n:
        for _ in range(e2e_steps):
            rc = L.deft4cu_optimise_batch(pp, lens, n, merge, e2e_res)
            assert rc == 0, N.last_error()
            out["d2h"] = sum(r.out_len for r in e2e_res) + C.sizeof(N.Result) * n
            L.deft4cu_free_results(e2e_res, n)
        torch.cuda.synchronize()
    out["e2e_s"] = (time.perf_counter() - t0) / e2e_steps
    ctx.barrier()
    return out


def verify_stream(raw, opt, r):
    """The rewritten stream inflates to exactly the bytes the input inflates to, and the device's length / CRC-32 /
    Adler-32 are theirs (incremental, so a 2.8 GB inflate never sits in memory twice)."""
    def digest(data):
        d = zlib.decompressobj(-15)
        crc, ad, n = 0, 1, 0
        for off in range(0, len(data), 1 << 24):
            chunk = d.decompress(data[off:off + (1 << 24)])
            crc, ad, n = zlib.crc32(chunk, crc), zlib.adler32(chunk, ad), n + len(chunk)
        chunk = d.flush()
        crc, ad, n = zlib.crc32(chunk, crc), zlib.adler32(chunk, ad), n + len(chunk)
        assert d.eof, "stream does not end with a final block"
        return crc & 0xffffffff, ad & 0xffffffff, n
    want = digest(raw)
    got = digest(opt)
    assert got == want, ("rewritten stream inflates differently", got, want)
    assert (r.crc32, r.adler32, r.uncompressed_len) == want, ("device checksums differ", (r.crc32, r.adler32, r.uncompressed_len), want)
    assert len(opt) * 8 - 7 <= r.size_bits_out <= len(opt) * 8, (len(opt), r.size_bits_out)
    assert len(opt) <= len(raw)
    # saved_bits is the reference's own running count (DeflateStream.java:519,565); with stored blocks it follows the
    # drifting `pos` (SURVEY.md H5), so it is reported, not asserted
    return r.size_bits_in - r.size_bits_out - r.saved_bits


DUMP_BYTES = 1 << 23     # output bytes kept by dump_outputs (32 MB as float32)
DUMP_SEED = 0xD4D0


def dump_outputs(path, N, res):
    """Write what a caller of the timed path receives for every stream, in stream order, as float64 `<field>.npy`
    (every field of deft4cu_result except the output buffer itself), plus `out_crc32.npy` (CRC-32 of each output
    stream: covers every byte) and `out_bytes.npy` (float32).  `out_bytes` is all output streams concatenated when they
    hold at most DUMP_BYTES bytes, otherwise the bytes at the sorted positions
    np.random.default_rng(DUMP_SEED).integers(0, total_length, DUMP_BYTES): the same positions whenever the total
    length is the same."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    views = [np.ctypeslib.as_array(r.out, (r.out_len,)) if r.out_len else np.zeros(0, np.uint8) for r in res]
    for name, _ in N.Result._fields_:
        if name != "out":
            np.save(os.path.join(path, name + ".npy"), np.array([getattr(r, name) for r in res], dtype=np.float64))
    np.save(os.path.join(path, "out_crc32.npy"), np.array([zlib.crc32(v) for v in views], dtype=np.float64))
    starts = np.cumsum([0] + [len(v) for v in views])
    total = int(starts[-1])
    if total <= DUMP_BYTES:
        pos = np.arange(total)
    else:
        pos = np.sort(np.random.default_rng(DUMP_SEED).integers(0, total, DUMP_BYTES))
    sample = np.empty(len(pos), np.float32)
    bounds = np.searchsorted(pos, starts)
    for k, v in enumerate(views):
        lo, hi = bounds[k], bounds[k + 1]
        sample[lo:hi] = v[pos[lo:hi] - starts[k]]
    np.save(os.path.join(path, "out_bytes.npy"), sample)


def roofline_of(m, peak, peak_src):
    algo = m["in_bytes"] + m["out_bytes"] + 2 * m["unc_bytes"]      # DESIGN.md: A = C_in + C_out + 2 U per pass
    opt_ms = m["fam"][3]
    achieved = algo / (opt_ms / 1e3) / 1e9 if opt_ms > 0 else 0.0
    return {"bound": "hbm", "kernel": "k_opt_blocks", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": algo,
            "kernel_ms": opt_ms, "family_ms_per_step": dict(zip(FAMILIES, m["fam"]))}


def run_shapes(ctx, L, N, a, peak, peak_src):
    """Short runs of the other named shapes: ONE list per shape, the same on every rank, dealt to the ranks by
    deft4j_b200.sharding.shard_streams (strong scaling; no collective on the data path)."""
    import workloads as W
    from deft4j_b200.sharding import shard_streams
    cores = os.cpu_count() or 1
    shapes = {}
    plan = [("c3_png_idat", lambda: W.c3_streams(768, first=10_000), 1, "768 synthetic 256x256 RGBA PNG IDAT streams, merge blocks"),
            ("c4_zip_entries", lambda: W.c4_streams(768, seed=5), 1, "768 ZIP-entry payloads (stored / Z_FIXED / dynamic, 1-256 KiB), merge blocks"),
            ("c5_adversarial", lambda: W.c5_streams(scale=8), 1, "15 adversarial streams: len-258 dist-1 / dist-32768 at 8 MiB, sparse alphabets; merge blocks"),
            ("c2_reference_sample", lambda: reference_sample("c2", cores, a.sample_seconds)[0], 0,
             "exactly the streams the CPU reference arm is timed on (same_config), --no-merge-blocks like the headline")]
    for name, gen, merge, what in plan:
        t0 = time.time()
        streams = gen()
        shards = shard_streams([len(s) for s in streams], ctx.world)
        mine = [streams[i] for i in shards[ctx.rank]]
        m = measure(ctx, L, N, mine, merge, steps=3, warmup=4, verify=not a.no_verify, e2e_steps=2)
        dev_ms = ctx.max(m["dev_ms"]) / 3
        e2e_s = ctx.max(m["e2e_s"])
        total_in = sum(len(s) for s in streams)
        fams = ctx.gather(m["fam"])
        rf = roofline_of({"in_bytes": ctx.sum(m["in_bytes"]), "out_bytes": ctx.sum(m["out_bytes"]),
                          "unc_bytes": ctx.sum(m["unc_bytes"]), "fam": [max(f[k] for f in fams) for k in range(8)]}, peak, peak_src)
        shapes[name] = {"workload": what, "streams": len(streams), "input_bytes": total_in, "merge_blocks": bool(merge),
                        "value": total_in / (dev_ms / 1e3) / 1e6, "e2e": total_in / e2e_s / 1e6, "unit": "MB/s",
                        "ms_per_step": dev_ms, "scaling": "strong", "frac": rf["frac"],
                        "family_ms_per_step": rf["family_ms_per_step"], "saved_bits": ctx.sum(m["saved_bits"]),
                        "uncompressed_bytes": ctx.sum(m["unc_bytes"]),
                        "output_verified": None if a.no_verify else bool(m["verified"]), "seconds": round(time.time() - t0, 1)}
    shapes["c3_png_files"] = run_png_files(ctx, a)
    shapes["c4_zip_file"] = run_zip_file(ctx, a)
    return shapes


def run_zip_file(ctx, a, count=768):
    """C4 through the container layer: ONE ZIP archive per rank with method-8 entries (stored / Z_FIXED / dynamic deflate
    payloads) -> deft4cu_zip_optimise_batch (native archive model, the entries as one device batch) -> rewritten archive
    in host memory; wall clock around the C-ABI call (`e2e`), around the Python API that also copies the result into
    `bytes` (`e2e_python_api`) and around the Python mirror of ZipFile (`python_mirror_e2e`: read_containers ->
    optimise_containers -> write).  The ZIP model restates the un-vendored lljzip reader (parity unpinned); the entries'
    streams are c4_zip_entries', split over the ranks."""
    import io
    import zipfile
    import workloads as W
    from deft4j_b200.container import read_containers, optimise_containers, optimise_zip_files
    from deft4j_b200.container._front import front_call
    t0 = time.time()
    per = max(1, count // ctx.world)
    arch = W.c4_zip_archive(per, seed=5 + ctx.rank)

    def abi_call():
        L_, r_, n_ = front_call("deft4cu_zip_optimise_batch", [arch], True)
        L_.deft4cu_free_file_results(r_, n_)

    def native():
        return optimise_zip_files([arch], True)

    def mirror():
        conts = read_containers([arch], ["c4.zip"])
        assert conts[0] is not None
        saved = optimise_containers(conts, True)[0]
        return [{"status": 0, "out": conts[0].write(), "saved_bits": saved}]

    def timed(fn, passes, warm):
        best, res = None, None
        for it in range(warm + passes):
            ctx.barrier()
            t = time.perf_counter()
            res = fn()
            dt = ctx.max(time.perf_counter() - t)
            if it >= warm:
                best = dt if best is None else min(best, dt)
        return best, res

    best_abi, _ = timed(abi_call, 3, 3)
    best, res = timed(native, 2, 1)
    best_py, res_py = timed(mirror, 2, 1)
    out = res[0]["out"]
    assert res[0]["status"] == 0
    ok = None
    if not a.no_verify:
        assert out == res_py[0]["out"], "native front-end and Python mirror disagree"
        zi, zo = zipfile.ZipFile(io.BytesIO(arch)), zipfile.ZipFile(io.BytesIO(out))
        assert zo.testzip() is None and len(zo.infolist()) == per
        for i in zi.infolist()[::max(1, per // 64)]:
            assert zo.read(i.filename) == zi.read(i.filename), i.filename
        assert len(out) <= len(arch)
        ok = True
    total_in = ctx.sum(len(arch))
    return {"workload": "one ZIP archive of %d method-8 entries per rank through the native ZIP front-end "
                        "(deft4cu_zip_optimise_batch): read, optimise (merge blocks), write" % per,
            "entries": per * ctx.world, "input_bytes": total_in, "merge_blocks": True, "e2e": total_in / best_abi / 1e6,
            "unit": "MB/s", "seconds_per_pass": best_abi, "e2e_python_api": total_in / best / 1e6,
            "python_mirror_e2e": total_in / best_py / 1e6, "saved_bits": ctx.sum(res[0]["saved_bits"]),
            "output_bytes": ctx.sum(len(out)), "scaling": "strong", "output_verified": ok, "seconds": round(time.time() - t0, 1)}


def run_png_files(ctx, a, count=768):
    """C3 through the container layer (SURVEY.md 8 'next' row: PNGFile): PNG files in host memory ->
    deft4cu_png_optimise_batch (native chunk model on host threads, all IDAT streams one device batch) -> rewritten
    files in host memory; wall clock around the call, host bytes in and out.  Compare with c3_png_idat.e2e (the same
    images as bare streams).  `python_mirror_e2e` is the same work through the Python mirror of PNGFile
    (read_containers -> optimise_containers -> write), which the CLI uses for mixed folders."""
    import io
    import workloads as W
    from deft4j_b200.container import read_containers, optimise_containers, optimise_png_files
    t0 = time.time()
    files = W.c3_png_files(count, first=10_000)
    mine = files[ctx.rank::ctx.world]
    names = ["img%d.png" % i for i in range(len(mine))]

    def native():
        return optimise_png_files(mine, True)

    def mirror():
        conts = read_containers(mine, names)
        assert all(c is not None for c in conts)
        saved = optimise_containers(conts, True)
        return [{"status": 0, "out": c.write(), "saved_bits": s} for c, s in zip(conts, saved)]

    def timed(fn, passes, warm):
        best, res = None, None
        for it in range(warm + passes):
            ctx.barrier()
            t = time.perf_counter()
            res = fn()
            dt = ctx.max(time.perf_counter() - t)
            if it >= warm:
                best = dt if best is None else min(best, dt)
        return best, res

    from deft4j_b200.container.png_file import _png_call

    def abi_call():     # the C-ABI call alone, as the raw-stream e2e is timed: host buffers in, library-owned host buffers out
        L_, r_, n_ = _png_call(mine, True, None)
        L_.deft4cu_free_file_results(r_, n_)

    best_abi, _ = timed(abi_call, 4, 3)
    best, res = timed(native, 3, 1)
    best_py, res_py = timed(mirror, 2, 2)
    assert all(r["status"] == 0 for r in res)
    ok = None
    if not a.no_verify:
        from PIL import Image
        assert [r["out"] for r in res] == [r["out"] for r in res_py], "native front-end and Python mirror disagree"
        for k in range(0, len(mine), max(1, len(mine) // 16)):
            assert Image.open(io.BytesIO(res[k]["out"])).tobytes() == Image.open(io.BytesIO(mine[k])).tobytes(), "pixels differ"
            assert len(res[k]["out"]) <= len(mine[k])
        ok = True
    total_in = sum(len(f) for f in files)
    return {"workload": "%d Pillow-written 256x256 RGBA PNG files (compress_level=6) through the native PNG front-end "
                        "(deft4cu_png_optimise_batch): read, optimise (merge blocks), write; wall clock around the C-ABI call "
                        "(e2e), around deft4j_b200.container.optimise_png_files which also copies the files into Python bytes "
                        "(e2e_python_api), and around the Python mirror of PNGFile (python_mirror_e2e)" % count,
            "files": count, "input_bytes": total_in, "merge_blocks": True, "e2e": total_in / best_abi / 1e6, "unit": "MB/s",
            "seconds_per_pass": best_abi, "e2e_python_api": total_in / best / 1e6, "python_mirror_e2e": total_in / best_py / 1e6,
            "saved_bits": ctx.sum(sum(r["saved_bits"] for r in res)), "output_bytes": ctx.sum(sum(len(r["out"]) for r in res)),
            "scaling": "strong", "output_verified": ok, "seconds": round(time.time() - t0, 1)}


def run_ours(a):
    ctx = Ctx()
    from deft4j_b200 import _native as N
    L = N.lib()
    name, merge = workload_config(a)
    t_gen = time.time()
    streams = make_streams(a, ctx.rank)
    t_gen = time.time() - t_gen
    dump = a.dump_outputs
    if dump and ctx.world > 1:
        dump = os.path.join(dump, "rank%d" % ctx.rank)
    m = measure(ctx, L, N, streams, merge, a.steps, a.warmup, sample_clocks=True, verify=not a.no_verify, dump=dump)
    dev_ms = ctx.max(m["dev_ms"])
    total_in = ctx.sum(m["in_bytes"])
    value = total_in * a.steps / (dev_ms / 1e3) / 1e6
    e2e_value = total_in / ctx.max(m["e2e_s"]) / 1e6
    peak, peak_src = peaks()
    roofline = roofline_of(m, peak, peak_src)
    # DRAM traffic of the dominant kernel comes from an ncu capture (never measured inside a timed run):
    # profiles/traffic.json records dram__bytes_read.sum + dram__bytes_write.sum of one k_opt_blocks launch and the input
    # size it was captured on; it is reported as `traffic` only when this run's launch processes the same input.
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if abs(tj.get("input_bytes", 0) - m["in_bytes"]) <= 0.01 * m["in_bytes"] and tj.get("merge_blocks", 0) == merge:
            roofline["traffic"] = tj["dram_bytes"]
        roofline["traffic_note"] = tj
    except Exception:
        pass
    per_rank = ctx.gather({"rank": ctx.rank, "ms_per_step": m["dev_ms"] / a.steps, "e2e_s_per_step": m["e2e_s"],
                           "family_ms_per_step": dict(zip(FAMILIES, m["fam"]))})
    shapes = None
    if a.workload == "c2" and not a.no_shapes:
        shapes = run_shapes(ctx, L, N, a, peak, peak_src)
    if ctx.rank == 0:
        base = None
        if ctx.world == 1 and not a.no_cpu:
            base = run_cpu_baseline(a, merge, a.sample_seconds)
        in_bytes = m["in_bytes"]
        cfg = {"workload": name, "merge_blocks": bool(merge), "streams_per_gpu": m["n"], "input_bytes_per_gpu": in_bytes,
               "uncompressed_bytes_per_gpu": m["unc_bytes"], "saved_bits_per_gpu": m["saved_bits"],
               "l2": "inputs larger than L2" if in_bytes > (126 << 20) else
               "inputs smaller than L2; every step re-parses from HBM-resident input after the previous step's "
               "multi-GB intermediates passed through L2", "datagen_s": round(t_gen, 1)}
        if a.workload == "c2" and not merge:
            cfg["merge_note"] = C2_WHY_NO_MERGE
        line = {"metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": ctx.world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": cfg, "clocks": m["clocks"], "gpu_launches": m["launches"],
                "e2e": {"value": e2e_value, "unit": "MB/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": m["d2h"]},
                "roofline": roofline, "output_verified": bool(m["verified"]) if not a.no_verify else None,
                "verify": m["verified"], "saved_bits": m["saved_bits"], "per_rank": per_rank}
        if shapes is not None:
            line["shapes"] = shapes
        if base:
            line["cpu_baseline"] = base
        print(json.dumps(line))
    if ctx.dist:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
