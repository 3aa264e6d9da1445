"""The candidate engine at its edges (run on the B200): the explicit LZ77 shapes of tests/lz_streams.py against the
oracle - bytes, saved bits, consumed bytes, checksums, the block model, and for shapes under 50 000 symbols every
candidate's size - plus properties that need no oracle and so run at full size: position independence inside a batch,
one large stream among many small ones, and the stress build of the engine's caches and queues."""
import ctypes as C
import functools
import os
import subprocess
import sys
import zlib

import pytest

import lz_streams as Z
import workloads as W
from test_gpu_parity import _oracle_batch, _split_calls, compare_stream

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRACE_MAX_SYMBOLS = 50_000


@pytest.fixture(scope="module")
def gpu():
    import deft4j_b200
    from deft4j_b200 import _native
    _native.lib()  # raises when the CUDA library or a device is missing: no fallback
    return deft4j_b200


@functools.lru_cache(maxsize=None)
def _edge():
    return Z.edge_shapes()


@functools.lru_cache(maxsize=None)
def _big():
    return Z.big_shapes()


EDGE_NAMES = (["nm%d" % n for n in Z.MATCH_COUNTS] +
              ["merge_a%d_nm%d" % (a, n) for a in (31, 33) for n in (33, 257, 2049)] +
              ["length_bins", "tile_geometry", "sparse_tiles", "blocked_literals", "zero_cost_fixed", "queue_overflow",
               "queue_long_overflow", "stored_65535", "stored_65536", "deep_codes"])


@pytest.mark.parametrize("merge", [False, True])
@pytest.mark.parametrize("name", EDGE_NAMES)
def test_edge_shape_matches_oracle(gpu, oracle, name, merge):
    compare_stream(gpu, oracle, _edge()[name].raw, merge)


def trace_compare(gpu, oracle, raw):
    """every candidate of every optimiseBlock call, (index, size), as in test_candidate_trace_matches_oracle"""
    from deft4j_b200 import _native
    CAP = 3_000_000
    OL, GL = oracle.lib(), _native.lib()
    OL.ora_trace_begin.argtypes = [C.POINTER(C.c_int64), C.c_size_t]
    OL.ora_trace_end.restype = C.c_size_t
    o = oracle.OracleDeflateStream()
    assert o.parse(raw)
    buf = (C.c_int64 * (2 * CAP))()
    OL.ora_trace_begin(buf, CAP)
    so = o.optimise(False)
    n = OL.ora_trace_end()
    assert n < CAP
    # The device prices the stored form only when it lays the stream out (the stored size depends on the block's bit
    # position), so its per-block rounds follow the reference's only while no Huffman block is won by the stored form:
    # the traced shapes are chosen so.
    assert all(o.blockInfo(i).type != 0 for i in range(o.blockCount())), "a traced shape must not end in a stored block"
    ref = _split_calls([(buf[2 * i], buf[2 * i + 1]) for i in range(n)])
    g = gpu.DeflateStream()
    assert g.parse(raw)
    assert GL.deft4cu_debug_trace_begin(CAP) == 0
    sg = g.optimise(False)
    gbuf = (C.c_int64 * (2 * CAP))()
    gn = C.c_uint32(0)
    assert GL.deft4cu_debug_trace_end(gbuf, CAP, C.byref(gn)) == 0
    assert gn.value < CAP
    got = _split_calls([(gbuf[2 * i], gbuf[2 * i + 1]) for i in range(gn.value)])
    assert sg == so
    assert len(got) == len(ref), (len(got), len(ref))
    for call, ((ri, rc), (gi, gc)) in enumerate(zip(ref, got)):
        assert ri == gi, (call, "incumbent")
        assert gc, call
        for idx, sz in gc.items():
            assert rc.get(idx) == sz, (call, idx, rc.get(idx), sz)
        assert max(gc) <= max(rc) and len(rc) - len(gc) <= 56 * 4 * 16, (call, len(rc), len(gc))
        # the chosen candidate: the first strict minimum over the oracle's full list is in the device's list too
        best = min(rc.values())
        first = min(i for i, v in rc.items() if v == best)
        if best < ri:
            assert gc.get(first) == best, (call, first)
    assert g.asBytes() == o.asBytes()


TRACE_NAMES = [n for n in EDGE_NAMES if n not in ("deep_codes", "stored_65535", "stored_65536")]


@pytest.mark.parametrize("name", TRACE_NAMES)
def test_edge_shape_candidate_trace(gpu, oracle, name):
    s = _edge()[name]
    assert sum(b.n for b in s.blocks) < TRACE_MAX_SYMBOLS
    trace_compare(gpu, oracle, s.raw)


def _compare_results(streams, res, ref):
    for k, (raw, r, (saved, out, consumed, crc, adler, ulen)) in enumerate(zip(streams, res, ref)):
        assert r["status"] == 0, k
        assert (r["saved_bits"], r["consumed"]) == (saved, consumed), k
        assert r["out"] == out, k
        assert (r["crc32"], r["adler32"], r["uncompressed_len"]) == (crc, adler, ulen), k


def test_big_weight_shapes_match_oracle(gpu, oracle):
    """Blocks of more than 4 MiB on both sides of the exact-weight threshold, merge off and on (the oracle runs in a
    process pool), and every candidate of the block whose removal of a length symbol leaves a literal of weight > 2^22."""
    big = _big()
    names = sorted(big)
    streams = [big[n].raw for n in names]
    for merge in (False, True):
        ref = _oracle_batch(streams, merge)
        for raw, (saved, out, consumed, crc, adler, ulen) in zip(streams, ref):
            r = gpu.optimise_batch([raw], merge)[0]
            _compare_results([raw], [r], [(saved, out, consumed, crc, adler, ulen)])
    trace_compare(gpu, oracle, big["big_weights_run"].raw)


# ---- full-size properties: no oracle -------------------------------------------------------------------------------------
def _key(r):
    return (r["status"], r["saved_bits"], r["out"], r["crc32"])


def _lead_stream(k):
    """a stream that decodes to exactly k bytes (a fixed block of literals)"""
    bw = W.BitWriter()
    W.fixed_block(bw, [0x61 + (i % 7) for i in range(k)], True)
    return bw.done()


@functools.lru_cache(maxsize=None)
def _large_streams():
    def deflate(data):
        co = zlib.compressobj(6, zlib.DEFLATED, -15, 9)
        return co.compress(data) + co.flush()
    import numpy as np
    n = 64 << 20
    period = np.random.default_rng(5).integers(0, 256, 32768, dtype="uint8").tobytes()
    return [W.c2_stream(16 << 20), deflate(b"\x41" * n), deflate((period * (n // 32768 + 1))[:n])]


def test_results_do_not_depend_on_the_position_in_the_batch(gpu, monkeypatch):
    """The 16 MiB C2 stream and the 64 MiB C5 shapes (blocks over 4 MiB: the exact-weight tree) alone, then behind
    streams that decode to k bytes, k = 1..15, 511, 512, 513: the blocks' decoded starts move through every residue mod
    16 and across a tile; with the slab poisoned, with one CTA per SM, and run twice."""
    big = _large_streams()
    alone = [_key(gpu.optimise_batch([raw], False)[0]) for raw in big]
    assert all(a[0] == 0 for a in alone)
    for k in list(range(1, 16)) + [511, 512, 513]:
        lead = [_lead_stream(k)]
        res = gpu.optimise_batch(lead + big, False)
        assert [_key(r) for r in res[len(lead):]] == alone, k
    batch = [_lead_stream(7)] + big
    first = [_key(r) for r in gpu.optimise_batch(batch, False)]
    assert first[1:] == alone
    assert [_key(r) for r in gpu.optimise_batch(batch, False)] == first
    monkeypatch.setenv("D4_POISON", "1")
    assert [_key(r) for r in gpu.optimise_batch(batch, False)] == first
    monkeypatch.delenv("D4_POISON")
    monkeypatch.setenv("D4_CTAS_PER_SM", "1")
    assert [_key(r) for r in gpu.optimise_batch(batch, False)] == first


def test_one_large_stream_among_many_small_ones(gpu):
    """Merge on: the merge phase sizes every CTA's scratch for the largest stream, so one 16 MiB stream among 300 small
    ones must not make the batch fail; every stream's result equals its result without the others (the large one and
    the first 30 small ones alone, the small ones also as a batch of their own)."""
    large = W.c2_stream(16 << 20)
    small = W.c3_streams(300, first=3000)
    res = gpu.optimise_batch([large] + small, True)
    assert all(r["status"] == 0 for r in res)
    assert _key(res[0]) == _key(gpu.optimise_batch([large], True)[0])
    assert [_key(r) for r in res[1:]] == [_key(r) for r in gpu.optimise_batch(small, True)]
    for raw, r in zip(small[:30], res[1:31]):
        assert _key(r) == _key(gpu.optimise_batch([raw], True)[0])
    assert zlib.decompress(res[0]["out"], -15) == zlib.decompress(large, -15)


# ---- the stress build: tiny queues and caches, forced exact-weight trees -------------------------------------------------
_STRESS_SCRIPT = r"""
import io, sys, zlib
sys.path.insert(0, %(root)r); sys.path.insert(0, %(tests)r)
import workloads as W, oracle_lib, lz_streams as Z
from conftest import GOLDEN_PAIRS, read_golden
import deft4j_b200
from deft4j_b200.container import getContainerForBytes
for inp, gold, merge in GOLDEN_PAIRS:
    data = read_golden(inp)
    cont = getContainerForBytes(data, inp, deft4j_b200.DeflateStream)
    assert cont.read(data)
    cont.optimise(merge, io.StringIO())
    assert cont.write() == read_golden(gold), inp
co = zlib.compressobj(6, zlib.DEFLATED, -15, 8)
streams = [co.compress(W.c2_text(300000)) + co.flush()] + [s.raw for s in Z.edge_shapes().values()]
for merge in (False, True):
    res = deft4j_b200.optimise_batch(streams, merge)
    for k, (raw, r) in enumerate(zip(streams, res)):
        o = oracle_lib.OracleDeflateStream(); assert o.parse(raw)
        assert r["status"] == 0, k
        assert r["saved_bits"] == o.optimise(merge) and r["out"] == o.asBytes(), (k, merge)
print("STRESS-OK")
"""


def test_engine_stress_build(gpu):
    """libdeft4cu_stress.so: histogram queues of 40 / 8 entries, two literal-cost arrays and two sign-mask slots (evicted
    all the time), three literal sets before the reset, and the exact-weight tree for every block.  The reference goldens,
    a C2 stream and every edge shape must come out as the oracle's."""
    lib = os.path.join(ROOT, "deft4j_b200", "libdeft4cu_stress.so")
    assert os.path.exists(lib), "run __graft_entry__.build()"
    env = dict(os.environ, DEFT4CU_LIB=lib)
    p = subprocess.run([sys.executable, "-c", _STRESS_SCRIPT % {"root": ROOT, "tests": os.path.join(ROOT, "tests")}],
                       env=env, capture_output=True, text=True, timeout=1200)
    assert p.returncode == 0 and "STRESS-OK" in p.stdout, p.stdout[-2000:] + p.stderr[-4000:]
