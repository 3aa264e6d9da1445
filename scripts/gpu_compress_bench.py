"""Device compressor benchmark (deft4cu_compress_batch): input MB/s, the time of the compressor (match + parse + emit)
against the whole one-shot call, and the output size against Python's zlib at levels 1, 6 and 9.

Inputs: C2 text (workloads.c2_text) at 256 MiB, the filtered scanlines of C3 images (the inflated IDAT streams of
workloads.c3_streams) at about 256 MiB, and 64 MiB of random bytes (every block ends up stored).  Every output is
inflated and compared with its input.  Times are a host clock around calls that end in a device synchronise, after a
warm-up call on the same input.  The card's name and power limit are read in the same run; the JSON goes to
profiles/ (or --out)."""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import workloads as W  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return "unknown (%r)" % e, "unknown"


def c3_scanlines(target):
    out, k = [], 0
    total = 0
    while total < target:
        raws = [zlib.decompress(s, -15) for s in W.c3_streams(64, first=k)]
        out += raws
        total += sum(map(len, raws))
        k += 64
    return out


def run(name, datas, merge, steps):
    import deft4j_b200
    from deft4j_b200 import DeflateStream
    total = sum(map(len, datas))
    res = deft4j_b200.compress_batch(datas, merge)   # warm-up
    t_one, t_comp = [], []
    for _ in range(steps):
        t0 = time.perf_counter()
        res = deft4j_b200.compress_batch(datas, merge)
        t_one.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        hs = DeflateStream.compress_batch(datas)      # upload + match + parse + emit + model set-up
        t_comp.append(time.perf_counter() - t0)
        del hs
    out = sum(len(r["out"]) for r in res)
    for d, r in zip(datas, res):
        assert r["status"] == 0 and zlib.decompress(r["out"], -15) == d, name
    z = {lvl: sum(len(zlib.compress(d, lvl)) - 6 for d in datas) for lvl in (1, 6, 9)}   # raw deflate: no zlib wrapper
    one, comp = min(t_one), min(t_comp)
    row = {"input": name, "streams": len(datas), "bytes": total, "merge": merge, "one_shot_s": one,
           "input_MBps": total / one / 1e6, "compressor_s": comp, "optimise_write_checksums_s": one - comp,
           "out_bytes": out, "zlib1_bytes": z[1], "zlib6_bytes": z[6], "zlib9_bytes": z[9],
           "ratio_vs_zlib1": out / z[1], "ratio_vs_zlib6": out / z[6], "ratio_vs_zlib9": out / z[9]}
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=256)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "compress_bench.json"))
    a = ap.parse_args()
    name, power = card()
    rows = []
    rows.append(run("c2_text", [W.c2_text(a.mib << 20)], False, a.steps))
    rows.append(run("c3_scanlines", c3_scanlines(a.mib << 20), False, a.steps))
    rows.append(run("random", [np.random.default_rng(1).integers(0, 256, (a.mib // 4) << 20, dtype=np.uint8).tobytes()],
                    False, a.steps))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"gpu": name, "power_limit": power, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
