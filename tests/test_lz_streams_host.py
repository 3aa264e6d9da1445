"""The explicit LZ77 stream generator (tests/lz_streams.py): every shape inflates to the bytes it claims, the oracle
parses it into exactly the intended symbol lists, and it has the properties it is named for."""
import functools
import zlib

import pytest

import lz_streams as Z


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


def test_shape_list_is_complete():
    assert sorted(_edge()) == sorted(EDGE_NAMES)


def _check_parse(oracle, s):
    assert zlib.decompress(s.raw, -15) == s.data
    o = oracle.OracleDeflateStream()
    assert o.parse(s.raw) and o.consumed == len(s.raw)
    assert o.getUncompressedData() == s.data
    assert o.blockCount() == len(s.blocks)
    for i, b in enumerate(s.blocks):
        info = o.blockInfo(i)
        assert info.type == (1 if b.kind == "fixed" else 2)
        assert info.n_symbols == b.n and info.uncompressed_len == b.ulen
        assert o.blockSymbols(i) == Z.oracle_symbols(b.syms), i
        if b.kind != "fixed":
            assert o.blockCodelens(i, 0)[:len(b.L)] == b.L[:len(o.blockCodelens(i, 0))], i


@pytest.mark.parametrize("name", EDGE_NAMES)
def test_edge_shape_parses_as_intended(oracle, name):
    _check_parse(oracle, _edge()[name])


def test_traced_shapes_stay_small():
    """every shape but the three largest is small enough for the candidate-by-candidate comparison"""
    for name, st in _edge().items():
        if name not in ("deep_codes", "stored_65535", "stored_65536"):
            assert sum(b.n for b in st.blocks) < 50_000, name


@pytest.mark.parametrize("nm", Z.MATCH_COUNTS)
def test_match_count_shapes(nm):
    s = _edge()["nm%d" % nm]
    assert s.blocks[-1].nm == nm
    assert all(b.nm % 32 for b in s.blocks[:-1]) and len(s.blocks) == 3


@pytest.mark.parametrize("a", [31, 33])
def test_merge_shapes_shift_ranks_inside_mask_words(a):
    for nm in (33, 257, 2049):
        s = _edge()["merge_a%d_nm%d" % (a, nm)]
        assert [b.nm for b in s.blocks] == [a, nm]   # the union's ranks of block B start at a: not a word boundary


def test_length_bins_shape():
    s = _edge()["length_bins"]
    b = s.blocks[0]
    lens = [m[0] for _, m in b.matches]
    dists = [m[1] for _, m in b.matches]
    bins = {}
    for l in lens:
        bins[Z.len_sym(l)] = bins.get(Z.len_sym(l), 0) + 1
    used = sorted(bins)
    assert used[0] == 257 and used[-1] == 285 and len(used) == 26
    empty = [k for k in range(257, 286) if k not in bins]
    assert empty and all(used[0] < k < used[-1] for k in empty)      # empty bins between used ones
    assert 32 in bins.values() and 33 in bins.values()              # one full and one split work item
    for k in used:
        base = Z.W._LEN_BASE[k - 257]
        top = 258 if k == 285 else min(257, base + (1 << Z.W._LEN_EB[k - 257]) - 1)
        ls = {l for l in lens if Z.len_sym(l) == k}
        assert base in ls and (top in ls or bins[k] < 2), k
    for d in range(30):
        base = Z.W._DIST_BASE[d]
        assert base in dists and base + (1 << Z.W._DIST_EB[d]) - 1 in dists, d
    assert 32768 in dists
    one = s.blocks[1]
    assert one.nm == 700 and {Z.len_sym(m[0]) for _, m in one.matches} == {263}   # one bin holds every match


def test_tile_geometry_shape():
    s = _edge()["tile_geometry"]
    assert sorted(b.residue for b in s.blocks) == list(range(16))
    for b in s.blocks:
        assert 0 in b.start_offsets and 511 in b.start_offsets
        assert b.ending_at_tile_end >= 1
        assert b.crossing_offsets == list(range(255, 512))   # from 254 a 258-byte match ends at the tile's end
        assert b.empty_tiles
    assert all(b.empty_run_boundaries for b in s.blocks)
    sp = _edge()["sparse_tiles"].blocks[0]
    assert len(sp.empty_run_boundaries) >= 5
    # literal runs longer than 1 024 bytes
    for b in s.blocks:
        run, best = 0, 0
        for x in b.syms:
            run = run + 1 if isinstance(x, int) else 0
            best = max(best, run)
        assert best > 1024


def test_literal_cost_shapes():
    b = _edge()["blocked_literals"].blocks[1]
    assert b.blocked >= 300 and b.blocked < b.nm
    z = _edge()["zero_cost_fixed"].blocks[0]
    assert z.zero >= 1500
    assert sum(1 for x in z.dc if x is not None and x < 0) >= 200 and sum(1 for x in z.dc if x is not None and x > 0) >= 200
    # 3 x 8 bits of literals against 7 (symbol 257) + 5 + 11 / 12 / 13 extra bits
    for (_, (length, dist)), x in zip(z.matches, z.dc):
        assert x == (1 if dist <= 8192 else 0 if dist <= 16384 else -1)


def test_queue_overflow_shapes():
    """The first replace pass over the block's own table replaces more matches than the histogram queue holds: more than
    HQS in all and more than HQL long ones (in the second shape all of them fit the main queue, so more than HQL long
    ones reach the long queue whatever the order of the warps)."""
    b = _edge()["queue_overflow"].blocks[0]
    assert b.replaced > Z.HQS and b.replaced_long > Z.HQL
    b = _edge()["queue_long_overflow"].blocks[0]
    assert b.replaced <= Z.HQS and b.replaced_long > Z.HQL
    assert b.L[ord("a")] == 1 and b.L[ord("b")] == 2
    # the rule recomputed by hand for one long match: 25 literals of 'a' / 'b' against 7 + 2 + 15 + 13 bits
    (_, (length, dist)), p = b.matches[0], b.mstart[0]
    lc = sum(b.L[x] for x in _edge()["queue_long_overflow"].data[p:p + length])
    assert b.dc[0] == lc - (7 + Z.len_ebits(length)) - (15 + 13) and dist > 16384


def test_stored_and_deep_code_shapes():
    a, b = _edge()["stored_65535"].blocks[0], _edge()["stored_65536"].blocks[0]
    assert (a.ulen, a.stored_ok, b.ulen, b.stored_ok) == (65535, True, 65536, False)
    d = _edge()["deep_codes"].blocks[0]
    for lens in (d.L, d.D):
        assert max(lens) == 15 and len({11, 12, 13, 14, 15} & set(lens)) >= 4


@pytest.mark.slow
def test_big_weight_shapes(oracle):
    """ulen + n + 4 lands on 2^22 - 1 and on 2^22 exactly (n counts the EOB, as k_emit counts a block's symbols); the
    third shape holds a literal that occurs more than 2^22 times once its length symbol is removed."""
    big = _big()
    lo, at, run = big["big_weights_below"].blocks[0], big["big_weights_at"].blocks[0], big["big_weights_run"].blocks[0]
    assert lo.ulen + lo.n + 4 == (1 << 22) - 1 and not lo.big_weights
    assert at.ulen + at.n + 4 == 1 << 22 and at.big_weights
    assert run.big_weights and run.ulen + run.n + 4 < 1 << 23
    assert big["big_weights_run"].data.count(b"a") > 1 << 22 and run.n < 50_000
    for s in big.values():
        _check_parse(oracle, s)
