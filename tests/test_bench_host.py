"""Host-side pieces of bench.py that the GPU box only exercises on one branch: the clock sampler's `nvidia-smi` fallback
(the box has the NVML module, so its runs take the in-process path)."""
import datetime
import os
import sys
import tempfile
import time

from conftest import ROOT

sys.path.insert(0, ROOT)


def test_clock_sampler_fallback_uses_only_samples_after_the_mark():
    import bench
    s = bench.ClockSampler.__new__(bench.ClockSampler)
    s.nv = None
    s.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)

    class Done:
        def terminate(self): pass
        def wait(self): pass
        def poll(self): return 0
    s.p = Done()
    now = time.time()

    def line(t, mhz, power_cap):
        ts = datetime.datetime.fromtimestamp(t).strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]
        return "%s, %d, 1965, 500.0, 0x0, Not Active, Not Active, Not Active, %s\n" % (ts, mhz, "Active" if power_cap else "Not Active")
    s.f.write(line(now - 5.0, 1200, True))      # warm-up sample: ignored
    s.f.write(line(now + 0.2, 1950, False))
    s.f.write(line(now + 0.7, 1965, False))
    s.f.write("garbage line\n")
    s.t_mark = now
    r = s.stop()
    assert r["samples"] == 2 and r["sm_mhz"] == 1957.5 and r["sm_max_mhz"] == 1965 and r["reasons"] == []
    assert not os.path.exists(s.f.name)


def test_dump_outputs_writes_every_result_field(tmp_path, monkeypatch):
    import ctypes as C
    import zlib
    import numpy as np
    import bench
    from deft4j_b200 import _native as N
    outs = [bytes(range(256)) * 3, b"", b"\x07" * 500, bytes(range(255, -1, -1))]
    bufs = [(C.c_uint8 * max(1, len(o))).from_buffer_copy(o.ljust(1, b"\0")) for o in outs]
    res = (N.Result * len(outs))()
    for k, (o, b) in enumerate(zip(outs, bufs)):
        res[k].status, res[k].saved_bits, res[k].crc32, res[k].size_bits_in = k % 2, 1000 * k - 1, 0xffffffff - k, 1 << 40
        res[k].out, res[k].out_len = (C.cast(b, C.POINTER(C.c_uint8)) if o else None), len(o)
    whole = b"".join(outs)
    bench.dump_outputs(str(tmp_path / "all"), N, res)
    d = {p.stem: np.load(p) for p in (tmp_path / "all").iterdir()}
    assert set(d) == {f for f, _ in N.Result._fields_ if f != "out"} | {"out_crc32", "out_bytes"}
    assert d["out_bytes"].dtype == np.float32 and (d["out_bytes"] == np.frombuffer(whole, np.uint8)).all()
    assert d["saved_bits"].dtype == np.float64 and list(d["saved_bits"]) == [-1, 999, 1999, 2999]
    assert list(d["crc32"]) == [0xffffffff - k for k in range(4)] and list(d["size_bits_in"]) == [1 << 40] * 4
    assert list(d["out_len"]) == [len(o) for o in outs] and list(d["status"]) == [0, 1, 0, 1]
    assert list(d["out_crc32"]) == [zlib.crc32(o) for o in outs]
    # larger than the budget: a seeded sample at sorted positions of the concatenated streams, the same every time
    monkeypatch.setattr(bench, "DUMP_BYTES", 300)
    bench.dump_outputs(str(tmp_path / "a"), N, res)
    bench.dump_outputs(str(tmp_path / "b"), N, res)
    a, b = np.load(tmp_path / "a" / "out_bytes.npy"), np.load(tmp_path / "b" / "out_bytes.npy")
    pos = np.sort(np.random.default_rng(bench.DUMP_SEED).integers(0, len(whole), 300))
    assert (a == b).all() and (a == np.frombuffer(whole, np.uint8)[pos]).all()


def test_clock_sampler_without_any_tool():
    import bench
    c = bench.ClockSampler(0)
    c.wait_ready(0.1)
    c.mark()
    r = c.stop()
    assert "sm_mhz" in r and "reasons" in r
