"""The device compressor (deft4cu_compress_batch, DeflateStream.compress_batch, `gzip-compress`).

CPU: the host restatement of the parse rule (deft4j_b200/csrc/lzrule.cuh, compiled into hosttest.cu) against a pure-Python
statement of the rule, its block layout, and the oracle.  GPU: the device's fixed-coded stream F against the host's byte
for byte, and the one-shot results against the oracle and against the optimiser run on F."""
import ctypes as C
import functools
import gzip
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import hosttest_lib
import oracle_lib
import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_B = 32768


# ---- the rule in plain Python (workloads.fixed_block writes the blocks) ------------------------------------------------
def _py_compress(d, B=DEFAULT_B):
    n = len(d)
    prev, head = [-1] * n, {}
    for p in range(n - 2):
        h = ((d[p] << 10) ^ (d[p + 1] << 5) ^ d[p + 2]) & 0x7FFF
        prev[p] = head.get(h, -1)
        head[h] = p

    def match(p, e):
        if p + 3 > n:
            return None
        cap = min(258, e - p)
        best, bestd, q, k = 0, 0, prev[p], 0
        while k < 32 and q >= 0 and p - q <= 32768:
            ln = 0
            while ln < cap and d[q + ln] == d[p + ln]:
                ln += 1
            if ln > best:
                best, bestd = ln, p - q
            q, k = prev[q], k + 1
        if best < 3 or (best == 3 and bestd > 4096):
            return None
        return best, bestd

    bw = W.BitWriter()
    starts = list(range(0, n, B)) or [0]
    for k, s in enumerate(starts):
        e = min(n, s + B)
        M = [match(p, e) for p in range(s, e)] + [None]
        syms, i = [], s
        while i < e:
            m, mn = M[i - s], M[i + 1 - s]
            if m and (i + 1 == e or (mn[0] if mn else 0) <= m[0]):
                syms.append(m)
                i += m[0]
            else:
                syms.append(d[i])
                i += 1
        W.fixed_block(bw, syms, k == len(starts) - 1)
    return bw.done()


def host_compress(d, B=DEFAULT_B):
    L = hosttest_lib.lib()
    L.host_lz_compress.restype = C.c_longlong
    L.host_lz_compress.argtypes = [C.c_char_p, C.c_uint64, C.c_uint32, C.c_char_p, C.c_uint64]
    cap = len(d) * 2 + 1024
    buf = C.create_string_buffer(cap)
    bits = L.host_lz_compress(bytes(d), len(d), B, buf, cap)
    assert bits >= 0
    return buf.raw[:(bits + 7) // 8]


def _rand(n, seed):
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8).tobytes()


@functools.lru_cache(maxsize=None)
def inputs():
    """name -> (data, block size): the shapes the rule has edges at."""
    r = _rand(32769, 1)
    out = {
        "empty": (b"", DEFAULT_B), "one": (b"a", DEFAULT_B), "two": (b"ab", DEFAULT_B), "three": (b"abc", DEFAULT_B),
        "run258": (b"z" * 258, DEFAULT_B), "run259": (b"z" * 259, DEFAULT_B), "run100000": (b"\x41" * 100000, DEFAULT_B),
        "period32768": ((r[:32768] * 4)[:100000], DEFAULT_B), "period32769": ((r * 4)[:100000], DEFAULT_B),
        "dist4096": (b"xyz" + _rand(4093, 2) + b"xyz" + _rand(500, 3), DEFAULT_B),
        "dist4097": (b"xyz" + _rand(4094, 2) + b"xyz" + _rand(500, 3), DEFAULT_B),
        "multiple_b256": (W.c2_text(256 * 12), 256), "multiple_b32768": (W.c2_text(65536), DEFAULT_B),
        "random": (_rand(70000, 4), DEFAULT_B),
    }
    for B in (256, 1000, 32768, 65535):
        out["c2_b%d" % B] = (W.c2_text(70000, seed=7), B)
    return out


SMALL = 4200   # the pure-Python statement is compared on the inputs up to about this size


@pytest.mark.parametrize("name", sorted(inputs()))
def test_host_rule_layout_and_roundtrip(name):
    d, B = inputs()[name]
    f = host_compress(d, B)
    assert zlib.decompress(f, -15) == d
    o = oracle_lib.OracleDeflateStream()
    assert o.parse(f)
    nblk = max(1, -(-len(d) // B))
    assert o.blockCount() == nblk
    for k in range(nblk):
        bi = o.blockInfo(k)
        assert bi.type == 1 and bi.uncompressed_len <= B
    if len(d) <= SMALL:
        assert f == _py_compress(d, B)


def test_host_rule_matches_python_on_small_text():
    for B in (256, 1000, DEFAULT_B):
        d = W.c2_text(4096, seed=11)
        assert host_compress(d, B) == _py_compress(d, B)
    d = _rand(3000, 9) * 2
    assert host_compress(d) == _py_compress(d)


@pytest.mark.parametrize("merge", [False, True])
@pytest.mark.parametrize("name", sorted(inputs()))
def test_oracle_optimises_host_stream(name, merge):
    d, B = inputs()[name]
    if merge and len(d) > 64 << 10:
        pytest.skip("the merge cascade is quadratic on long stationary inputs; merge is checked up to 64 KiB")
    o = oracle_lib.OracleDeflateStream()
    assert o.parse(host_compress(d, B))
    o.optimise(merge)
    assert zlib.decompress(o.asBytes(), -15) == d


def test_compress_batch_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from deft4j_b200 import _native, compress_batch, DeflateStream
    with pytest.raises(_native.Deft4cuError):
        compress_batch([b"abc"])
    with pytest.raises(_native.Deft4cuError):
        DeflateStream.compress_batch([b"abc"])


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    import deft4j_b200
    from deft4j_b200 import _native
    _native.lib()  # raises when the CUDA library or a device is missing: no fallback
    return deft4j_b200


def _device_F(gpu, datas, B=0):
    return [s.asBytes() for s in gpu.DeflateStream.compress_batch(datas, block_bytes=B)]


def _oracle_opt(f, merge):
    o = oracle_lib.OracleDeflateStream()
    assert o.parse(f)
    saved = o.optimise(merge)
    return o.asBytes(), saved


@functools.lru_cache(maxsize=None)
def _c3_raw():
    return [zlib.decompress(s, -15) for s in W.c3_streams(3)]


@pytest.mark.gpu
def test_device_F_equals_host(gpu):
    for name, (d, B) in sorted(inputs().items()):
        assert _device_F(gpu, [d], B) == [host_compress(d, B)], name
    big = W.c2_text(8 << 20)
    assert _device_F(gpu, [big]) == [host_compress(big)]
    for B in (256, 4096, 32768, 65535):
        raws = _c3_raw()
        assert _device_F(gpu, raws, B) == [host_compress(x, B) for x in raws], B


@pytest.mark.gpu
def test_one_shot_matches_oracle(gpu):
    for name, (d, B) in sorted(inputs().items()):
        f = host_compress(d, B)
        for merge in (False, True):
            if merge and len(d) > 64 << 10:
                continue
            r = gpu.compress_batch([d], merge, B)[0]
            out, saved = _oracle_opt(f, merge)
            assert r["status"] == 0, name
            assert (r["out"], r["saved_bits"]) == (out, saved), (name, merge)
            assert r["size_bits_in"] == oracle_lib_bits(f) and r["consumed"] == len(d) == r["uncompressed_len"]


def oracle_lib_bits(f):
    o = oracle_lib.OracleDeflateStream()
    assert o.parse(f)
    return o.getSizeBits()


@pytest.mark.gpu
def test_64mib_text_equals_optimise_of_F(gpu):
    d = W.c2_text(64 << 20)
    r = gpu.compress_batch([d], False)[0]
    f = _device_F(gpu, [d])[0]
    ref = gpu.optimise_batch([f], False)[0]
    assert r["out"] == ref["out"] and r["saved_bits"] == ref["saved_bits"]
    assert zlib.decompress(r["out"], -15) == d
    assert r["crc32"] == zlib.crc32(d) & 0xffffffff and r["adler32"] == zlib.adler32(d) & 0xffffffff
    assert r["uncompressed_len"] == len(d)
    assert len(r["out"]) <= len(zlib.compress(d, 1))


def _mixed(count, seed=3):
    rng = np.random.default_rng(seed)
    text = W.c2_text(4 << 20, seed=seed)
    out = []
    for k in range(count):
        n = 0 if k % 50 == 0 else int(np.exp(rng.uniform(0, np.log(200 << 10))))
        off = int(rng.integers(0, len(text) - n))
        out.append(text[off:off + n])
    # streams that end and begin with the same bytes: a window leaking across streams would find matches
    tail = text[:5000]
    out += [tail, tail, tail[:3], tail]
    return out


@pytest.mark.gpu
def test_batch_equals_one_call_each(gpu):
    from deft4j_b200 import _native
    datas = _mixed(496)
    L = _native.lib()
    before = L.deft4cu_debug_engine_launches()
    res = gpu.compress_batch(datas, True)
    assert L.deft4cu_debug_engine_launches() == before + 1
    for d, r in zip(datas, res):
        one = gpu.compress_batch([d], True)[0]
        assert r == one
        assert zlib.decompress(r["out"], -15) == d


@pytest.mark.gpu
def test_regrouped_with_parsed_handles(gpu):
    datas = _mixed(12, seed=8)
    zs = []
    for x in (W.c2_text(30000, seed=1), W.c2_text(70000, seed=2)):
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        zs.append(co.compress(x) + co.flush())
    for merge in (False, True):
        alone = []
        for d in datas:
            s = gpu.DeflateStream.compress_batch([d])[0]
            s.optimise(merge)
            alone.append(s.asBytes())
        for z in zs:
            s = gpu.DeflateStream.parse_batch([z])[0]
            s.optimise(merge)
            alone.append(s.asBytes())
        # compressed handles from two batches, parsed handles from two batches, in one list
        hs = gpu.DeflateStream.compress_batch(datas[:6]) + gpu.DeflateStream.compress_batch(datas[6:])
        hs += gpu.DeflateStream.parse_batch(zs[:1]) + gpu.DeflateStream.parse_batch(zs[1:])
        gpu.DeflateStream.optimise_batch(hs, merge)
        assert [s.asBytes() for s in hs] == alone
        # compressed handles only (regrouped into one compressed batch)
        hs = [gpu.DeflateStream.compress_batch([d])[0] for d in datas]
        gpu.DeflateStream.optimise_batch(hs, merge)
        assert [s.asBytes() for s in hs] == alone[:len(datas)]


@pytest.mark.gpu
def test_split_past_the_decoded_limit(gpu, monkeypatch):
    datas = _mixed(40, seed=5)
    ref = gpu.compress_batch(datas, False)
    monkeypatch.setenv("D4_MAX_DECODED", str(300 << 10))
    assert gpu.compress_batch(datas, False) == ref


_BUILD_SCRIPT = r"""
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(tests)r)
import hashlib, workloads as W
import deft4j_b200
d = W.c2_text(3 << 20, seed=21)
r = deft4j_b200.compress_batch([d], True, 0)[0]
print(hashlib.sha256(r["out"]).hexdigest(), r["saved_bits"])
"""


@pytest.mark.gpu
def test_stress_builds_give_identical_bytes(gpu):
    outs = []
    for lib in ("libdeft4cu.so", "libdeft4cu_smallpools.so", "libdeft4cu_stress.so"):
        env = dict(os.environ, DEFT4CU_LIB=os.path.join(ROOT, "deft4j_b200", lib))
        p = subprocess.run([sys.executable, "-c", _BUILD_SCRIPT % {"root": ROOT, "tests": os.path.join(ROOT, "tests")}],
                           env=env, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
        outs.append(p.stdout.strip())
    assert outs[0] == outs[1] == outs[2]


@pytest.mark.gpu
def test_gzip_compress_cli(gpu, tmp_path):
    from deft4j_b200 import _native
    from deft4j_b200.__main__ import main
    d = W.c2_text(300000, seed=4) + _rand(20000, 6)
    src = tmp_path / "in.txt"
    src.write_bytes(d)
    for extra in ([], ["--merge-blocks"], ["--block-bytes", "1000"]):
        dst = tmp_path / ("out%d.gz" % len(extra))
        assert main(["gzip-compress", str(src), str(dst)] + extra) == 0
        assert gzip.decompress(dst.read_bytes()) == d
    L = _native.lib()
    res = (_native.Result * 1)()
    ptrs, lens = _native.make_ptr_arrays([d])
    for bad in (255, 65536):
        assert L.deft4cu_compress_batch(ptrs, lens, 1, 0, bad, res) == _native.ERR_ARG
    with pytest.raises(_native.Deft4cuError):
        gpu.compress_batch([d], True, 100)
