"""CPU pin of the enumeration's items (deft4j_b200/csrc/enum.cuh sweep_item / join, compiled as host code): the kernel's
sweepers take the items of a sweep from a queue in whatever order they get to them, and every item of the selection
sweep selects inside its own candidates.  Whatever the order, the discovery sweeps must raise the same requests at every
execute level, and the join of the items' records must select exactly what one walk over the items in order selects."""
import ctypes as C
import zlib

import numpy as np
import pytest

import test_host_enum as E
import workloads as W

WALK, FORWARD, REVERSE, SHUFFLE = -1, 0, 1, 2
ORDERS = [(FORWARD, 0), (REVERSE, 0), (SHUFFLE, 1), (SHUFFLE, 0x9E3779B97F4A7C15)]


def _lib():
    L = E._engine()
    L.host_engine_order.argtypes = [C.c_void_p, C.c_int, C.c_ulonglong]
    L.host_engine_selection.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
    L.host_engine_reqlog.restype = C.c_size_t
    L.host_engine_reqlog.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong), C.c_size_t]
    return L


def _blocks(oracle, raw):
    o = oracle.OracleDeflateStream()
    assert o.parse(raw)
    data = o.getUncompressedData()
    blocks, pos = [], 0
    for i in range(o.blockCount()):
        bi = o.blockInfo(i)
        blk = {"type": bi.type, "ulen": bi.uncompressed_len, "data": data[pos:pos + bi.uncompressed_len], "payload": bi.litlen_size_bits,
               "hbits": bi.header_size_bits, "ncl": bi.num_codelen_lens}
        pos += bi.uncompressed_len
        if bi.type != 0:
            blk["sym"] = o.blockSymbols(i)
            if bi.type == 2:
                blk["L"], blk["D"], blk["CL"] = o.blockCodelens(i, 0), o.blockCodelens(i, 1), o.blockCodelens(i, 2)
                blk["pairs"] = o.blockRlePairs(i)
        blocks.append(blk)
    return blocks


def _run_block(L, blk, order, seed, segmented):
    """Every optimiseBlock call of the block's rounds, in the given item order: per call the selection state, and the
    request log of the whole run."""
    h, keep = E._load(L, blk)
    L.host_engine_order(h, order, seed)
    calls = []
    try:
        for _ in range(64):
            res = (C.c_longlong * 16)()
            sel = (C.c_longlong * 7)()
            # a stored candidate one bit under the incumbent: it is the best at the head item until a later item beats it
            assert L.host_engine_round(h, -1, int(segmented), res, None, 0, None) == 0, list(res)
            incumbent = res[3]
            assert L.host_engine_round(h, incumbent - 1, int(segmented), res, None, 0, None) == 0, list(res)
            L.host_engine_selection(h, sel)
            calls.append(tuple(sel))
            assert L.host_engine_round(h, -1, int(segmented), res, None, 0, None) == 0, list(res)
            L.host_engine_selection(h, sel)
            calls.append(tuple(sel) + (res[15],))
            if res[0] >= incumbent:
                break
            L.host_engine_advance(h, 1)
        n = L.host_engine_reqlog(h, None, 0)
        log = (C.c_ulonglong * max(1, n))()
        L.host_engine_reqlog(h, log, n)
        return calls, list(log)[:n]
    finally:
        L.host_engine_free(h)


def _streams(oracle):
    raws = E._fixture_streams(oracle, "text.png", 3) + E._fixture_streams(oracle, "apng/ball.png", 2)
    raws += [E._deflate(W.c2_text(6000, seed=3), 6, zlib.Z_FIXED), E._deflate(W.c2_text(30_000, seed=4)),
             W.handmade_streams()["edge284"], W.handmade_streams()["dyn_partialflush_dyn"], W.handmade_streams()["rle_two_fixed"],
             E._deflate(bytes(range(256)) * 8), E._deflate(b"ab" * 3000 + bytes(range(64)))]
    raws += [s for s in W.c5_streams() if len(s) < 3000][:3]
    return raws


@pytest.mark.parametrize("mode", ["all", "segmented"])
def test_items_in_any_order_select_what_the_walk_selects(oracle, mode):
    L = _lib()
    checked = levels = 0
    for si, raw in enumerate(_streams(oracle)):
        for bi, blk in enumerate(_blocks(oracle, raw)):
            if blk["type"] == 0 or blk["ulen"] == 0:
                continue
            ref_calls, ref_log = _run_block(L, blk, WALK, 0, mode == "segmented")
            assert ref_log, (si, bi)
            for order, seed in ORDERS:
                calls, log = _run_block(L, blk, order, seed, mode == "segmented")
                # bestSize, bestIndex, bestStored, bestArg, restMin, sizeC1, candIndex (+ the materialised winner)
                assert calls == ref_calls, (si, bi, order, seed)
                assert log == ref_log, (si, bi, order, seed, "request sets per execute level")
            checked += len(ref_calls)
            levels += ref_log.count(2**64 - 1)
    assert checked > 40 and levels > 100, (checked, levels)


def test_a_stored_candidate_and_a_later_item_both_win_somewhere(oracle):
    """The probe calls above exercise both outcomes of the join: the head's stored candidate kept, and beaten later."""
    L = _lib()
    stored = beaten = 0
    for raw in _streams(oracle)[:6]:
        for blk in _blocks(oracle, raw):
            if blk["type"] == 0 or blk["ulen"] == 0:
                continue
            calls, _ = _run_block(L, blk, SHUFFLE, 7, False)
            for c in calls[0::2]:
                stored += c[2] == 1
                beaten += c[2] == 0 and c[1] != 0xFFFFFFFF
    assert stored > 0 and beaten > 0, (stored, beaten)
