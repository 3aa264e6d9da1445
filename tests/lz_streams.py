"""Explicit LZ77 streams for the candidate engine's edges (TEST INFRASTRUCTURE).

A stream is a list of blocks; a block is a list of symbols (an int literal or a (length, distance) pair) and a kind:
  ("fixed",)                      the fixed code;
  ("dynamic",)                    code lengths from oracle_lib.huffman_tree on the block's own frequencies (limit 15);
  ("explicit", litlen, dist)      the given code lengths.
`build` runs the copies itself, so the decoded bytes are known without an inflater, and writes the stream with
workloads.BitWriter / fixed_block / dynamic_block.  Every named shape returns a `Stream` whose per-block records carry the
properties the shape is meant to have (match count, start residue mod 16, tile crossings, what the first replace pass
replaces, ...), all computed here in Python, so that a CPU test can check that the shape really has them.
"""
import numpy as np

import oracle_lib
import workloads as W

DC_TILE = 512          # engine.cuh: decoded bytes per literal-cost tile
ENG_NW = 8             # engine.cuh: warps per CTA (ENG_NT 256)
HQS, HQL = 4608, 1024  # engine.cuh: histogram queue capacities of the product build
BIG_WEIGHTS = 1 << 22  # engine.cuh load_block: ulen + n + 4 at or above this takes the exact-weight tree
FIXED_L = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 6
FIXED_D = [5] * 30


def len_sym(length):
    return 285 if length == 258 else 257 + max(k for k in range(28) if W._LEN_BASE[k] <= length)


def dist_sym(dist):
    return max(k for k in range(30) if W._DIST_BASE[k] <= dist)


def len_ebits(length):
    return W._LEN_EB[len_sym(length) - 257]


def dist_ebits(dist):
    return W._DIST_EB[dist_sym(dist)]


def freqs(syms):
    """litlen (286, EOB included) and distance (30) frequencies of a symbol list"""
    fl, fd = [0] * 286, [0] * 30
    for s in syms:
        if isinstance(s, int):
            fl[s] += 1
        else:
            fl[len_sym(s[0])] += 1
            fd[dist_sym(s[1])] += 1
    fl[256] += 1
    return fl, fd


def huffman_lengths(freq):
    """the reference's length-limited tree (limit 15); a lone used symbol gets length 1 so the block stays decodable"""
    if sum(1 for f in freq if f) == 0:
        return [0] * len(freq)
    _, ln = oracle_lib.huffman_tree(list(freq), 15)
    return [l if f == 0 or l else 1 for f, l in zip(freq, ln)]


class BlockRec:
    """One block as written, with the properties the tests check."""

    def __init__(self, kind, syms, L, D, start, data):
        self.kind, self.syms, self.L, self.D, self.start = kind, syms, L, D, start
        self.matches = [(k, s) for k, s in enumerate(syms) if not isinstance(s, int)]
        self.nm = len(self.matches)
        self.n = len(syms) + 1                     # symbols the engine sees: the list plus its EOB
        self.ulen = sum(1 if isinstance(s, int) else s[0] for s in syms)
        self.residue = start % 16
        a0 = start & ~15
        # per match: decoded offset of its first byte, start inside its tile, end relative to that tile
        self.mstart, pos = [], start
        for s in syms:
            if not isinstance(s, int):
                self.mstart.append(pos)
            pos += 1 if isinstance(s, int) else s[0]
        self.tile_off = [(p - a0) % DC_TILE for p in self.mstart]
        mlen = [s[0] for _, s in self.matches]
        self.crossing = sum(1 for o, l in zip(self.tile_off, mlen) if o + l > DC_TILE)
        self.ending_at_tile_end = sum(1 for o, l in zip(self.tile_off, mlen) if o + l == DC_TILE)
        self.crossing_offsets = sorted({o for o, l in zip(self.tile_off, mlen) if o + l > DC_TILE and l == 258})
        self.start_offsets = set(self.tile_off)
        # tiles (as build_views / ensure_lit count them) that no match starts in, and the warps' tile runs
        ntiles = (start - a0 + self.ulen) // DC_TILE + 1
        per = (ntiles + ENG_NW - 1) // ENG_NW
        starts = {(p - a0) // DC_TILE for p in self.mstart}
        self.empty_tiles = [t for t in range(ntiles) if t not in starts]
        self.empty_run_boundaries = [t for t in self.empty_tiles if per and t % per == 0 and t > 0]
        # the cost-array entries under the block's own table (engine.cuh dc_val): literal cost of the copied bytes minus
        # the match's cost; None = a byte without a literal code (DC_BLOCKED)
        self.dc = []
        for (k, (length, dist)), p in zip(self.matches, self.mstart):
            lc = [L[b] for b in data[p:p + length]]
            if any(c == 0 for c in lc):
                self.dc.append(None)
                continue
            self.dc.append(sum(lc) - (L[len_sym(length)] + len_ebits(length)) - (D[dist_sym(dist)] + dist_ebits(dist)))
        self.blocked = sum(1 for x in self.dc if x is None)
        self.zero = sum(1 for x in self.dc if x == 0)
        rep = [i for i, x in enumerate(self.dc) if x is not None and x < 0]
        self.replaced = len(rep)                                      # what replaceBackrefs (no prune) turns into literals
        self.replaced_long = sum(1 for i in rep if mlen[i] > 24)      # ... of them, the ones hq_apply gives a warp each
        self.big_weights = self.ulen + self.n + 4 >= BIG_WEIGHTS
        self.stored_ok = self.ulen <= 65535


class Stream:
    def __init__(self, raw, data, blocks):
        self.raw, self.data, self.blocks = raw, data, blocks


def build(blocks):
    """blocks: [(kind, syms), ...] with kind ("fixed",) / ("dynamic",) / ("explicit", L, D) -> Stream"""
    out = bytearray()
    recs = []
    bw = W.BitWriter()
    for bi, (kind, syms) in enumerate(blocks):
        start = len(out)
        for s in syms:
            if isinstance(s, int):
                out.append(s)
            else:
                length, dist = s
                assert 3 <= length <= 258 and 1 <= dist <= 32768 and dist <= len(out), (bi, s, len(out))
                for _ in range(length):
                    out.append(out[-dist])
        final = bi == len(blocks) - 1
        if kind[0] == "fixed":
            W.fixed_block(bw, syms, final)
            L, D = FIXED_L, FIXED_D
        else:
            if kind[0] == "dynamic":
                fl, fd = freqs(syms)
                L, D = huffman_lengths(fl), huffman_lengths(fd)
            else:
                L, D = list(kind[1]), list(kind[2])
            L = L + [0] * (286 - len(L))
            D = D + [0] * (30 - len(D))
            nl = max(257, max(k for k in range(286) if L[k]) + 1)
            nd = max(1, max([k + 1 for k in range(30) if D[k]] or [1]))
            W.dynamic_block(bw, L[:nl], D[:nd], syms, final)
        recs.append(BlockRec(kind[0], syms, L, D, start, bytes(out)))
    return Stream(bw.done(), bytes(out), recs)


def oracle_symbols(syms):
    """the symbol list as OracleDeflateStream.blockSymbols spells it: (distance, literal or length, edge case)"""
    return [(0, s, 0) if isinstance(s, int) else (s[1], s[0], 0) for s in syms] + [(0, 256, 0)]


# ---- helpers that write symbol lists ------------------------------------------------------------------------------------
def _lits(rng, n, alphabet):
    return [int(x) for x in rng.choice(alphabet, n)]


def fill(n, dist=1):
    """n decoded bytes as few symbols as possible: matches of at most 258 bytes (distance `dist`), literals for a rest of
    one or two bytes"""
    out = []
    while n >= 3:
        k = min(n, 258)
        if n - k in (1, 2):
            k -= 3
        out.append((k, dist))
        n -= k
    out += [0x41] * n
    return out


def _ulen(syms):
    return sum(1 if isinstance(s, int) else s[0] for s in syms)


def text_with_matches(rng, nm, pos, alphabet=b"etaoinshr", maxdist=4000):
    """nm matches of mixed lengths and distances between short literal runs, starting at decoded position pos"""
    syms = []
    p = pos
    for _ in range(nm):
        k = int(rng.integers(0, 4))
        syms += _lits(rng, k, list(alphabet))
        p += k
        length = int(rng.choice([3, 3, 4, 5, 6, 8, 11, 17, 30, 70, 258]))
        dist = int(rng.integers(1, min(p, maxdist) + 1))
        syms.append((length, dist))
        p += length
    return syms


# ---- the named shapes ------------------------------------------------------------------------------------------------------
MATCH_COUNTS = [0, 1, 31, 32, 33, 255, 256, 257, 2047, 2048, 2049, 4608, 4609]


def match_count_stream(nm, prefix=(37, 70), seed=1):
    """blocks with `prefix` match counts (not multiples of 32), then a dynamic block with exactly nm matches"""
    rng = np.random.default_rng(seed * 1000 + nm)
    blocks, pos = [], 0
    head = _lits(rng, 300, list(b"etaoinshr"))
    for k, c in enumerate(prefix):
        syms = (head if k == 0 else []) + text_with_matches(rng, c, pos + (len(head) if k == 0 else 0))
        blocks.append((("fixed",) if k % 2 == 0 else ("dynamic",), syms))
        pos += _ulen(syms)
    syms = text_with_matches(rng, nm, pos) + _lits(rng, 5, list(b"etaoinshr"))
    if pos == 0:
        syms = head + text_with_matches(rng, nm, len(head))
    blocks.append((("dynamic",), syms))
    return build(blocks)


def length_bins_stream():
    """One dynamic block with every length symbol and every distance symbol at its base and its largest extra value;
    bins of 32 and 33 matches (a full and a split work item of the least pass) and empty bins between used ones.  A second
    block holds one bin only."""
    rng = np.random.default_rng(7)
    syms = _lits(rng, 32768, list(range(256)))
    counts = {}
    order = [257 + k for k in range(29)]
    for k, s in enumerate(order):
        counts[s] = [2, 32, 33, 1, 5][k % 5]
    for s in (262, 268, 275):
        counts[s] = 0                                     # empty bins between used ones
    pairs = []
    for s, c in counts.items():
        k = s - 257
        # the largest length of symbol 284 is 257: 258 is spelled with 285 (284 + 31 is the reference's edge case)
        lo, hi = W._LEN_BASE[k], (258 if k == 28 else min(257, W._LEN_BASE[k] + (1 << W._LEN_EB[k]) - 1))
        for i in range(c):
            pairs.append(lo if i % 2 == 0 else hi)
    dists = []
    for d in range(30):
        dists += [W._DIST_BASE[d], W._DIST_BASE[d] + (1 << W._DIST_EB[d]) - 1]
    for i, length in enumerate(pairs):
        syms += _lits(rng, 1, list(range(256)))
        syms.append((length, dists[i % len(dists)]))
    first = ("dynamic",), syms
    one_bin = [(9, int(d)) for d in rng.integers(1, 3000, 700)]   # every match has length symbol 263
    return build([first, (("dynamic",), _lits(rng, 40, list(b"xyz")) + one_bin)])


def _tile_geometry_block(r, pos, head, run_tile):
    """the symbols of block r of tile_geometry_stream, decoded start pos; a literal run of 1 100 bytes follows the
    crossing match that starts in tile run_tile - 1, so tiles run_tile and run_tile + 1 have no match start"""
    rng = np.random.default_rng(1100 + r)
    syms = list(head)
    a0 = pos & ~15
    cur = [pos + _ulen(syms)]

    def add(xs):
        syms.extend(xs)
        cur[0] += _ulen(xs)

    def to(o):   # decoded bytes up to tile offset o, mostly as matches
        need = (o - (cur[0] - a0)) % DC_TILE
        if need:
            add(fill(need, 1 + int(rng.integers(0, 300))) if need >= 3 else _lits(rng, need, list(b"ab")))

    for o in range(254, 512):
        to(o)
        t = (cur[0] - a0) // DC_TILE
        add([(258, 1 + int(rng.integers(0, 500)))])
        if t + 1 == run_tile:
            add(_lits(rng, 1100, list(range(256))))   # a literal run: tiles with no match start
    to(0); add([(5, 7)])                              # a match at tile offset 0
    to(511); add([(3, 9)])                            # ... and at 511 (crosses by two bytes)
    to(500); add([(12, 40)])                          # ends exactly at the tile's end
    to(256); add([(256, 300)])                        # ... and one of 256 bytes from the middle
    add(_lits(rng, 1100, list(range(256))))           # a long run at the end of the block
    add([(7, 3)])
    add(_lits(rng, (r + 1 - cur[0]) % 16, list(b"cd")))   # the next block starts at residue r + 1 mod 16
    return syms, cur[0]


def tile_geometry_stream():
    """Sixteen blocks whose decoded starts cover every residue mod 16.  In each, matches start at tile offsets 0 and 511,
    end exactly at a tile's end, and 258-byte matches cross from every offset 254..511 into the next tile; literal runs
    longer than 1 024 bytes leave tiles without a match start, one of them at the start of a warp's run of tiles
    (ensure_lit gives each of the 8 warps ceil(tiles / 8) tiles).  The whole stream stays under 50 000 symbols, so that
    every candidate of every block can be compared with the oracle's."""
    blocks = []
    pos = 0
    head = _lits(np.random.default_rng(11), 600, list(range(256)))
    for r in range(16):
        h = head if r == 0 else []
        # the warp runs depend on the block's tile count, which the run itself changes: try boundaries until one is empty
        syms, end = _tile_geometry_block(r, pos, h, -1)
        for k in range(1, 8):
            for per in range(max(1, ((end - (pos & ~15)) // DC_TILE + 1) // 8 - 1), 60):
                cand, cend = _tile_geometry_block(r, pos, h, k * per)
                ntiles = (cend - (pos & ~15)) // DC_TILE + 1
                if (ntiles + ENG_NW - 1) // ENG_NW == per:
                    syms, end = cand, cend
                    break
            else:
                continue
            break
        blocks.append((("dynamic",) if r % 3 else ("fixed",), syms))
        pos = end
    return build(blocks)


def sparse_tiles_stream():
    """A block that is one long literal run between a few matches: most tiles, and every warp-run boundary but the
    first, have no match start."""
    rng = np.random.default_rng(12)
    syms = _lits(rng, 100, list(b"pq")) + [(40, 3)] + _lits(rng, 9000, list(range(256))) + [(30, 2000), (258, 1)]
    return build([(("dynamic",), syms)])


def blocked_literals_stream():
    """Byte values that only occur inside matches of the second block have no literal code there (DC_BLOCKED): the
    matches that copy them can never be replaced, and neither can their length symbol be removed.  The first block's
    bytes are skewed (p ~ 1 / (k + 1)), so that a Huffman code beats the stored form there too."""
    rng = np.random.default_rng(13)
    w = 1.0 / np.arange(1, 257)
    first = [int(x) for x in rng.choice(256, 3000, p=w / w.sum())]
    syms = _lits(rng, 50, list(b"klmnop"))
    p = 3050
    for i in range(1200):
        k = int(rng.integers(0, 3))
        syms += _lits(rng, k, list(b"klmnop"))
        p += k
        if i % 3 == 0:
            m = (int(rng.choice([3, 4, 10, 40])), int(rng.integers(p - 2990, p - 100)))   # copies first-block bytes
        else:
            m = (int(rng.choice([3, 5, 6])), int(rng.integers(1, 40)))
        syms.append(m)
        p += m[0]
    return build([(("fixed",), first), (("dynamic",), syms)])


def zero_cost_fixed_stream():
    """A fixed block of length-3 matches over bytes 0..143: at distances 8193..12288 a match costs exactly its three
    literals (7 + 5 + 12 = 24 = 3 x 8), so the entry is zero and only the pruning pass replaces it; at 4097..8192 the
    match is cheaper (23 bits: entry +1), at 16385.. dearer (25 bits: entry -1, replaced by either pass)."""
    rng = np.random.default_rng(14)
    syms = _lits(rng, 16400, list(range(144)))
    for i in range(3000):
        if i % 4 == 0:
            syms += _lits(rng, 1, list(range(144)))
        d = int(rng.integers(8193, 12289)) if i % 3 else int(rng.choice([int(rng.integers(4097, 8193)), int(rng.integers(16385, 16400))]))
        syms.append((3, d))
    return build([(("fixed",), syms)])


def _two_letter_lengths():
    """explicit, complete code lengths: 'a' 1 bit, 'b' 2 bits, 'c', 'd', the EOB and every length symbol 7 bits;
    distance symbols 0..13 take 1..14 bits and 28, 29 (distances above 16 384) 15 bits"""
    L = [0] * 286
    L[ord("a")], L[ord("b")], L[ord("c")], L[ord("d")] = 1, 2, 7, 7
    for s in range(256, 286):
        L[s] = 7
    D = [k + 1 for k in range(14)] + [0] * 14 + [15, 15]
    return L, D


def queue_overflow_stream(n_short=6000, n_long=1500, seed=15):
    """Two-letter text with explicit code lengths under which every match is dearer than its literals: the first replace
    pass over the block's own table replaces n_short matches of 3 bytes and n_long of 25..30 bytes, all at distances
    above 16 384, in one pass (the histogram queue holds HQS = 4 608 and HQL = 1 024)."""
    rng = np.random.default_rng(seed)
    L, D = _two_letter_lengths()
    text = list(b"a" * 9 + b"b")      # mostly 'a': 25..30 literals cost less than a 37-bit long match
    syms = _lits(rng, 16400, text)
    p = 16400
    kinds = [3] * n_short + [25, 26, 27, 28, 29, 30] * (n_long // 6) + [25] * (n_long % 6)
    rng.shuffle(kinds)
    for length in kinds:
        k = int(rng.integers(0, 2))
        syms += _lits(rng, k, text)
        p += k
        syms.append((int(length), int(rng.integers(16385, min(p, 32768) + 1))))
        p += int(length)
    return build([(("explicit", L, D), syms)])


def big_weights_stream(side):
    """A fixed block of (258, 3) matches padded with literals so that ulen + n + 4 (n: symbols with the EOB) is exactly
    2^22 - 1 (side 0, fast tree) or 2^22 (side 1, exact-weight tree)."""
    # 2 * L + 259 * M + 5 = target, with L literals and M matches
    M = 16194 if side == 0 else 16193
    target = BIG_WEIGHTS - 1 + side
    L = (target - 5 - 259 * M) // 2
    assert 2 * L + 259 * M + 5 == target and L >= 3
    lits = [int(x) for x in np.random.default_rng(16).integers(0, 256, L)]
    return build([(("fixed",), lits[:3] + [(258, 3)] * M + lits[3:])])


def big_weights_run_stream():
    """Above the threshold with a literal that, once a length symbol is removed, occurs more than 2^22 times: a weight the
    fast tree's 22-bit keys cannot hold.  A fixed block of 16 257 matches (258, 1) over 'a' and ten digits 1 000 times
    each."""
    digits = [0x30 + (k % 10) for k in range(10000)]
    return build([(("fixed",), [ord("a")] + [(258, 1)] * 16257 + digits)])


def stored_threshold_stream(ulen):
    """incompressible bytes in one fixed block: stored is the cheapest encoding, allowed only up to 65 535 bytes"""
    lits = [int(x) for x in np.random.default_rng(17 + ulen).integers(0, 256, ulen)]
    return build([(("fixed",), lits)])


def deep_codes_stream():
    """Fibonacci-like frequencies: litlen and distance codes of 11..15 bits (the second level of the parser's lookup
    tables)"""
    rng = np.random.default_rng(18)
    fib = [1, 1]
    while len(fib) < 30:
        fib.append(fib[-1] + fib[-2])
    syms = _lits(rng, 24600, list(b"0123456789"))
    lit_counts = {0x61 + k: min(fib[k], 4000) for k in range(22)}
    dist_counts = {d: min(fib[29 - d], 2500) for d in range(30)}
    pool = [b for b, c in lit_counts.items() for _ in range(c)]
    dpool = [d for d, c in dist_counts.items() for _ in range(c)]
    rng.shuffle(pool)
    rng.shuffle(dpool)
    lens = [3, 4, 5, 7, 9, 12, 20, 40, 100, 258]
    p = 24600
    for k, d in enumerate(dpool):
        syms += pool[2 * k:2 * k + 2]
        p += len(pool[2 * k:2 * k + 2])
        lo, hi = W._DIST_BASE[d], W._DIST_BASE[d] + (1 << W._DIST_EB[d]) - 1
        syms.append((lens[k % len(lens)], int(rng.integers(lo, min(hi, p) + 1))))
        p += lens[k % len(lens)]
    syms += pool[2 * len(dpool):]
    return build([(("dynamic",), syms)])


def edge_shapes():
    """name -> Stream for the shapes the oracle finishes in well under a second"""
    out = {}
    for nm in MATCH_COUNTS:
        out["nm%d" % nm] = match_count_stream(nm)
    for a in (31, 33):
        for nm in (33, 257, 2049):
            out["merge_a%d_nm%d" % (a, nm)] = match_count_stream(nm, prefix=(a,), seed=2)
    out["length_bins"] = length_bins_stream()
    out["tile_geometry"] = tile_geometry_stream()
    out["sparse_tiles"] = sparse_tiles_stream()
    out["blocked_literals"] = blocked_literals_stream()
    out["zero_cost_fixed"] = zero_cost_fixed_stream()
    out["queue_overflow"] = queue_overflow_stream()
    out["queue_long_overflow"] = queue_overflow_stream(n_short=2500, n_long=1500, seed=16)
    out["stored_65535"] = stored_threshold_stream(65535)
    out["stored_65536"] = stored_threshold_stream(65536)
    out["deep_codes"] = deep_codes_stream()
    return out


def big_shapes():
    """name -> Stream for the blocks of more than 4 MiB (the oracle needs seconds for each)"""
    return {"big_weights_below": big_weights_stream(0), "big_weights_at": big_weights_stream(1),
            "big_weights_run": big_weights_run_stream()}
