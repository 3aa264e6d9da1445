// enum.cuh — the candidate enumerator of DeflateStream.optimiseBlock (DeflateStream.java:343-490) as a SYMBOLIC
// program over ids, separated from the data-parallel work it asks for.
//
// A candidate of the reference (a DeflateBlockHuffman copy) is determined by
//     mid    id of its symbol list  = bit mask "this match has been replaced by its literals" (common.cuh)
//     tabid  id of its code tables  (Tab, hash-consed)
//     hid    id of its dynamic header (Hdr: RLE pairs, header code, numCodelenLens, size)
//     payload = litlenSizeBits
// and every mutator of the reference is a pure function of those ids:
//     replace / least passes   (mid, tabid, op) -> (mid', payload delta)        DeflateBlockHuffman.java:222-319,373-458
//     recodeHuffman            mid -> (tabid, default hid, payload)               :670-743
//     recodeToFixedHuffman     mid -> payload                                     :637-653
//     header mutators          (hid, op) -> hid'                                  :471-476,579-635
//     56 header strategy trials  tabid -> (first-minimum bits, its index)         DeflateStream.java:277-316
// The reference's enumeration (multi -> run -> aor -> trials, the tie-break contract of SURVEY.md §8a) is walked over
// memo tables of those functions, cut into 17 items (the head and every (seed, variant)) that the lanes of a CTA
// take from a queue.  A miss whose inputs are known is queued as a request and poisons everything that depends on it;
// after the sweep the whole CTA computes the queued requests side by side (engine.cuh: Huffman trees of different
// requests in different warps, passes CTA-wide, header trials 28 threads per table) and the sweep is repeated, skipping
// the items that completed earlier.  The enumeration does not depend on which candidate is winning, so when a sweep
// raises no request a final sweep feeds every candidate to the selection callback (DeflateStream.java:349-368) with the
// reference's strict `<`: each item selects inside its own candidates and a join stitches the items back in the
// reference's order.
//
// The file compiles as host code too (D4_HOST_TEST): tests/test_host_units.py drives this very enumerator with a plain
// serial executor (hosttest.cu) against the oracle's candidate trace.
#pragma once
#include "huff.cuh"

namespace d4 {

#ifdef D4_HOST_TEST
#define D4_HD inline
#define D4_HD_BIG inline
// the host harness runs the sweeps one after the other
#define D4_CAS_U32(p, cmp, val) ((*(p) == (cmp)) ? (*(p) = (val), (cmp)) : *(p))
#define D4_ADD_I32(p, val) (*(p) += (val))
#define D4_OR_U32(p, val) (*(p) |= (val))
#define D4_OR_U64(p, val) (*(p) |= (val))
#else
#define D4_HD __device__ __forceinline__
#define D4_HD_BIG __device__ __noinline__
// several threads of a CTA sweep different parts of the enumeration at once
#define D4_CAS_U32(p, cmp, val) atomicCAS((p), (cmp), (val))
#define D4_ADD_I32(p, val) atomicAdd((p), (val))
#define D4_OR_U32(p, val) atomicOr((p), (val))
#define D4_OR_U64(p, val) atomicOr((p), (val))
#endif

#ifdef D4_SMALL_POOLS           // stress build: ordinary inputs overflow the pools, which forces the segmented rounds
constexpr int MAXM = 96, MAXT = 96, MAXH = 192, PMEMO = 256;
#else
constexpr int MAXM = 192;     // distinct symbol-list masks kept per block (a C2 block meets ~65 in its two rounds)
constexpr int MAXT = 256;     // distinct code tables kept per block
constexpr int MAXH = 512;     // dynamic headers kept per block
constexpr int PMEMO = 512;    // pass memo slots (open addressing)
#endif
constexpr int QPASS = 64, QREC = 24, QHDR = 64, QTRIAL = 64;
constexpr int TAB_FIXED = 0;  // tab id 0 is always the fixed code (HuffmanTable.java:166-209)

// ops of the pass memo
enum { OP_REPLACE = 0, OP_REPLACE_PRUNE = 1, OP_LEAST0 = 2, OP_LEAST1 = 3, OP_FIXED = 4 };
// header mutators
enum { HOP_RECODE = 0, HOP_RECODE_LESS = 1, HOP_OPT = 2 };
enum { ST_EMPTY = 0, ST_PENDING = 1, ST_DONE = 2 };

struct SC {                    // symbolic candidate
    short mid, tabid, hid;     // hid < 0: none (FIXED)
    signed char type;          // 1 FIXED, 2 DYNAMIC
    signed char ok;            // 0: depends on a request that has not been computed yet
    long long payload;
};

struct PSlot { unsigned key; unsigned short mid; unsigned short state; long long delta; };
struct RSlot { unsigned short tabid, hid; unsigned state; long long payload; };

// memo tables + request queues of one block (shared memory on the device)
struct SymState {
    PSlot pm[PMEMO];
    RSlot rc[MAXM];
    unsigned short hop[MAXH][3];      // 0 absent, 0xFFFF pending, else hid' + 1
    unsigned short hbits[MAXH];        // dynamicHeaderSizeBits of every header (< 14 + 57 + 320 * 14)
    unsigned short trialBits[MAXT];    // first-minimum header bits over the 56 strategies
    unsigned char trialArg[MAXT];
    unsigned char trialState[MAXT];
    // request lists of one execution step, compacted by the executor from the PENDING entries of the tables above
    unsigned short qPass[QPASS], qRec[QREC], qTrial[QTRIAL];
    unsigned short qHdr[QHDR];         // hid << 2 | op
    int nqPass, nqRec, nqHdr, nqTrial;
    int nP;                            // used pass memo slots
    int nMasks, nTabs, nHdrs;
    int overflow;                      // a pool filled up during this round
    unsigned doneItem;                 // items (Enumer::sweep_item) that completed in an earlier sweep of this round
    unsigned long long doneAor;        // ... and the bases (seed, variant, base) inside them
    int requested;                     // a sweep marked something PENDING since this was last cleared
};

D4_HD void sym_reset(SymState& S, int tid, int nthreads) {
    for (int k = tid; k < PMEMO; k += nthreads) { S.pm[k].key = 0; S.pm[k].state = ST_EMPTY; }
    for (int k = tid; k < MAXM; k += nthreads) S.rc[k].state = ST_EMPTY;
    for (int k = tid; k < MAXH * 3; k += nthreads) S.hop[k / 3][k % 3] = 0;
    for (int k = tid; k < MAXT; k += nthreads) S.trialState[k] = ST_EMPTY;
    if (tid == 0) {
        S.nqPass = S.nqRec = S.nqHdr = S.nqTrial = 0;
        S.nP = 0; S.nMasks = 0; S.nTabs = 0; S.nHdrs = 0; S.overflow = 0;
        S.doneItem = 0; S.doneAor = 0; S.requested = 0;
    }
}

D4_HD unsigned pm_key(int mid, int tabid, int op) { return 0x80000000u | ((unsigned)op << 24) | ((unsigned)tabid << 12) | (unsigned)mid; }
D4_HD int pm_key_mid(unsigned k) { return (int)(k & 0xFFF); }
D4_HD int pm_key_tab(unsigned k) { return (int)((k >> 12) & 0xFFF); }
D4_HD int pm_key_op(unsigned k) { return (int)((k >> 24) & 0x7F); }
// slot of `key`; when absent and `insert` is set the key is claimed (state PENDING) and *inserted tells so.  Returns -1
// when absent and not inserted.
D4_HD int pm_find(SymState& S, unsigned key, bool insert, bool* inserted) {
    unsigned x = key * 0x9E3779B1u;
    x ^= x >> 15;
    unsigned h = x & (PMEMO - 1);
    *inserted = false;
    while (true) {
        unsigned k = S.pm[h].key;
        if (k == 0) {
            if (!insert) return -1;
            if (S.nP >= PMEMO * 3 / 4) { S.overflow = 1; return -1; }
            k = D4_CAS_U32(&S.pm[h].key, 0u, key);
            if (k == 0) { S.pm[h].state = ST_PENDING; D4_ADD_I32(&S.nP, 1); *inserted = true; return (int)h; }
        }
        if (k == key) return (int)h;
        h = (h + 1) & (PMEMO - 1);
    }
}

// trace sink of the selection sweep (parity debugging): host tests pass a vector, the device a global buffer
struct TraceSink {
    long long* buf;
    unsigned cap;
    unsigned* n;
};

// items of one sweep (Enumer::sweep_item): the head, then (seed, variant, base) in the reference's order
constexpr int NITEMS = 1 + 4 * 4;
static_assert(NITEMS <= 32, "one done bit per item");

// selection outcome of one item swept apart (Enumer::put_item / join)
struct ItemRec {
    long long bestSize, restMin, sizeC1;
    SC best;
    unsigned bestIndex;    // inside the item's own candidates (0xffffffff: none beat the value carried in)
    unsigned candIndex;    // candidates the item counted
    int bestStored, bestArg;
};

struct Enumer {
    const int* trialAll;       // [tabid * 56 + k] header bits of every strategy (trace only; may be null)
    TraceSink* trace;          // null: no trace
    // the block
    SC B;
    int blockType;             // type of B
    bool storedOK;             // uncompressed length <= 65535: the stored candidate exists (DeflateStream.java:376-383)
    long long storedSize;      // < 0: not compared here (phase A resolves it in the replay)
    bool select;               // final sweep: every op is resolved, run the selection callback
    // sweep state
    bool poisoned;
    int internalError;
    // selection state (carried across the segments of a segmented round)
    long long bestSize, sizeI, sizeC1, restMin;
    int bestStored, bestArg;
    unsigned candIndex, bestIndex;
    SC best;

    // Everything below is inlined into ONE routine (sweep_item, a single copy) without calls (the sweep runs in a single thread next to CTAs that
    // stream through L1: a call stack in local memory would cost an L2 round trip per access).  `st` is the block's
    // memo state (shared memory on the device).

    // ---- memo access ---------------------------------------------------------------------------------------
    D4_HD SC bad(SC c) { c.ok = 0; poisoned = true; return c; }
    D4_HD long long size(const SymState& st, const SC& c) const { return c.payload + (c.type == 2 ? (long long)st.hbits[c.hid] : 0); }

    D4_HD_BIG SC op_pass(SymState& st, SC c, int op) {
        if (!c.ok) return bad(c);
        if (op >= OP_LEAST0 && op <= OP_LEAST1 && c.type != 2) return c;   // removeDistLitLeastExpensive: DYNAMIC only
        const unsigned key = pm_key(c.mid, c.tabid, op);
        bool ins;
        const int slot = pm_find(st, key, !select, &ins);
        if (slot >= 0 && !ins) {
            const PSlot& p = st.pm[slot];
            if (p.state != ST_DONE) return bad(c);
            c.mid = (short)p.mid;
            c.payload -= p.delta;
            return c;
        }
        if (select) internalError = 1;
        if (ins) st.requested = 1;
        return bad(c);
    }
    D4_HD_BIG SC op_recode(SymState& st, SC c) {   // recodeHuffman (:670-743)
        if (!c.ok) return bad(c);
        RSlot& r = st.rc[c.mid];
        if (r.state == ST_DONE) { c.tabid = (short)r.tabid; c.hid = (short)r.hid; c.payload = r.payload; c.type = 2; return c; }
        if (r.state == ST_EMPTY) {
            if (select) { internalError = 2; return bad(c); }
            r.state = ST_PENDING;
            st.requested = 1;
        }
        return bad(c);
    }
    D4_HD_BIG SC op_recode_less(SymState& st, SC c) { return op_recode(st, op_pass(st, c, OP_REPLACE_PRUNE)); }   // recodeHuffmanLessMatches (:655-658)
    D4_HD_BIG SC op_to_fixed(SymState& st, SC c) {   // recodeToFixedHuffman (:637-653)
        if (!c.ok) return bad(c);
        if (c.type == 1) return c;
        const unsigned key = pm_key(c.mid, 0xFFF, OP_FIXED);
        bool ins;
        const int slot = pm_find(st, key, !select, &ins);
        if (slot >= 0 && !ins) {
            const PSlot& p = st.pm[slot];
            if (p.state != ST_DONE) return bad(c);
            c.payload = p.delta; c.type = 1; c.tabid = TAB_FIXED; c.hid = -1;
            return c;
        }
        if (select) internalError = 3;
        if (ins) st.requested = 1;
        return bad(c);
    }
    D4_HD_BIG SC op_hdr(SymState& st, SC c, int hop) {
        if (!c.ok) return bad(c);
        if (c.type != 2) return c;
        volatile unsigned short& h = st.hop[c.hid][hop];
        if (h != 0 && h != 0xFFFF) { c.hid = (short)(h - 1); return c; }
        if (h == 0) {
            if (select) { internalError = 4; return bad(c); }
            h = 0xFFFF;
            st.requested = 1;
        }
        return bad(c);
    }
    // DeflateBlockHuffman.optimise (:460-469): replace pass, then the header half; *saved = bits saved
    D4_HD_BIG SC op_optimise(SymState& st, SC c, long long* saved) {
        if (!c.ok) return bad(c);
        const long long before = size(st, c);
        c = op_pass(st, c, OP_REPLACE);
        if (c.ok && c.type == 2) c = op_hdr(st, c, HOP_OPT);
        if (c.ok) *saved = before - size(st, c);
        return c;
    }

    // ---- selection callback (DeflateStream.java:349-368) ---------------------------------------------------
    D4_HD void trace_put(long long idx, long long sz) {
        if (!trace) return;
        const unsigned k = (*trace->n)++;
        if (k < trace->cap) { trace->buf[2 * k] = idx; trace->buf[2 * k + 1] = sz; }
    }
    D4_HD_BIG void cb(const SymState& st, const SC& c, bool isRest = true) {
        if (!c.ok) { poisoned = true; return; }
        if (!select) return;
        const long long sz = size(st, c);
        trace_put(candIndex, sz);
        if (isRest && sz < restMin) restMin = sz;
        if (sz < bestSize) { bestSize = sz; bestStored = 0; bestIndex = candIndex; best = c; bestArg = -1; }
        candIndex++;
    }
    // `o` = optimiseBlockNormal(t) (DeflateStream.java:319-327): a candidate only when it saved something
    D4_HD void cb_if_saved(const SymState& st, const SC& o, long long saved) {
        if (o.ok) { if (saved > 0) cb(st, o); } else poisoned = true;
    }

    // one base of addOptimisedRecoded's 56 header strategy trials (DeflateStream.java:277-316): the first-minimum
    // strategy is the only one the strict `<` of the callback can accept
    D4_HD_BIG void trial_base(SymState& st, const SC& c) {
        if (!c.ok) { poisoned = true; return; }
        const int t = c.tabid;
        if (st.trialState[t] != ST_DONE) {
            if (select) { internalError = 5; poisoned = true; return; }
            if (st.trialState[t] == ST_EMPTY) { st.trialState[t] = ST_PENDING; st.requested = 1; }
            return;
        }
        if (!select) return;
        if (trace && trialAll)
            for (int k = 0; k < 56; k++) trace_put(candIndex + k, c.payload + trialAll[t * 56 + k]);
        const long long sz = c.payload + st.trialBits[t];
        if (sz < restMin) restMin = sz;
        if (sz < bestSize) { bestSize = sz; bestStored = 0; bestIndex = candIndex + st.trialArg[t]; best = c; bestArg = st.trialArg[t]; }
        candIndex += 56;
    }

    // recodedHuffmanFull (DeflateStream.java:212-229): x is replaced while a further recodeHuffmanLessMatches shrinks it
    D4_HD_BIG SC recoded_full(SymState& st, SC x, bool* changed) {
        *changed = false;
        if (!x.ok) return bad(x);
        while (true) {
            const SC t = op_recode_less(st, x);
            if (!t.ok) return bad(x);
            if (size(st, t) >= size(st, x)) break;
            x = t;
            *changed = true;
        }
        return x;
    }

    enum { SEG_HEAD = 1, SEG_MULTI_H = 2, SEG_MULTI_O = 4, SEG_FIXED = 8, SEG_LEAST0 = 16, SEG_LEAST1 = 32, SEG_ALL = 63 };

    // start of a round (DeflateStream.optimiseBlock entry): the incumbent is B
    D4_HD void begin_round(SymState& st) {
        bestSize = size(st, B);
        bestStored = 0; bestArg = -1;
        sizeI = bestSize; sizeC1 = bestSize;
        restMin = 0x7fffffffffffffffll;
        candIndex = 0; bestIndex = 0xffffffffu;
        best = B;
        internalError = 0;
        st.doneItem = 0; st.doneAor = 0;
    }

    // DeflateStream.optimiseBlock (:343-490) is cut into NITEMS items that can be swept in any order and by several
    // threads at once.  The nesting is the reference's: runOptimisationsCallbackMulti (:443-463) over four seeds m,
    // runOptimisationsCallback (:400-442) over up to four variants r of a seed, addOptimisedRecoded (:265-317) over three
    // bases a of a variant.  Item 0 is the head (the optimised block and the stored candidate); item 1 + m * 4 + r is one
    // variant of one seed with its three bases, and the items in index order emit the reference's candidates in its order.
    // An item recomputes its prefix (the seed and the variant) through the memo tables; when the prefix is not known yet
    // the item is poisoned and asks for nothing beyond what the prefix asked for, so a sweep over all items raises exactly
    // the requests of one walk over the whole enumeration, whatever the order of the items.  Returns true when the item
    // met no missing or pending op (an item outside `seg`, or an r = 3 variant that recodedHuffmanFull left unchanged, is
    // empty and returns true).
    D4_HD bool sweep_item(SymState& st, bool sel, unsigned seg, int item) {
        select = sel;
        poisoned = false;
        const int m = (item - 1) >> 2, r = (item - 1) & 3;
        long long saved = 0;
        SC wO = B, wH = B;
        bool hasO = false;
        if (item == 0 || (m == 1 && blockType != 1)) { wO = op_optimise(st, B, &saved); hasO = wO.ok && saved > 0; }
        if (item == 0 && (seg & SEG_HEAD)) {
            if (sel) trace_put(-1, size(st, B));
            if (hasO) { cb(st, wO, false); if (sel) sizeC1 = size(st, wO); }
            if (storedOK && sel) {
                if (storedSize >= 0 && storedSize < bestSize) { bestSize = storedSize; bestStored = 1; bestIndex = candIndex; }
                candIndex++;
            }
        }
        if (blockType == 1) {   // a FIXED block is recoded first; multi(O) starts from the recode's optimised form
            wH = op_recode(st, B);
            if (item == 0 || m == 1) { wO = op_optimise(st, wH, &saved); hasO = wO.ok && saved > 0; }
        }
        if (item == 0) return !poisoned;
        // ---- the seed of this runOptimisationsCallbackMulti ------------------------------------------------------------
        SC wE;
        if (m == 0) { if (!(seg & SEG_MULTI_H)) return true; wE = wH; }
        else if (m == 1) { if (!(seg & SEG_MULTI_O)) return true; if (!hasO) return !poisoned; wE = wO; }
        else if (m == 2) {
            if (r == 0 && (seg & SEG_FIXED) && blockType != 1) {   // the fixed-code candidate sits between multi(O) and the least seeds
                long long s2 = 0;
                const SC F = op_optimise(st, op_to_fixed(st, wH), &s2);
                cb(st, F);
            }
            if (!(seg & SEG_LEAST0)) return !poisoned;
            wE = op_pass(st, wH, OP_LEAST0);
        } else { if (!(seg & SEG_LEAST1)) return true; wE = op_pass(st, wH, OP_LEAST1); }
        if (!wE.ok) { poisoned = true; return false; }
        // ---- the variant this runOptimisationsCallback works on -------------------------------------------------------
        SC wX = wE;
        if (r == 1) wX = op_recode(st, wE);
        else if (r >= 2) {
            wX = op_recode_less(st, wE);
            if (r == 3) {
                bool full = false;
                wX = recoded_full(st, wX, &full);
                if (wX.ok && !full) return !poisoned;
            }
        }
        if (!wX.ok) { poisoned = true; return false; }
        cb(st, wX);
        for (int a = 0; a < 3; a++) {
            SC wY;
            if (a == 0) {
                wY = op_hdr(st, wX, HOP_RECODE); cb(st, wY);                                  // post
                long long sv = 0;
                const SC o = op_optimise(st, wY, &sv); cb_if_saved(st, o, sv);             // post optimised
            } else wY = op_pass(st, wX, a == 1 ? OP_LEAST0 : OP_LEAST1);
            // ---- addOptimisedRecoded(y) ---------------------------------------------------------------------------------
            // the four bases are only ever read by the trials: their Tab and payload.  Every trial rewrites the header from
            // the Tab (optimiseBlockDynBlock -> rewriteHeader, DeflateStream.java:184-198), so the header half of
            // DeflateBlockHuffman.optimise() cannot influence any candidate here and is not run.
            const int an = (item - 1) * 3 + a;
            int nb = 0;
            if (select || !((st.doneAor >> an) & 1)) {   // a base that completed in an earlier sweep asks for nothing
                const bool outerA = poisoned;
                poisoned = false;
                const SC wB0 = op_pass(st, wY, OP_REPLACE);                               // optimiseBlockCopyHelper(toOptimise)
                const SC wB1 = op_pass(st, op_recode(st, wY), OP_REPLACE);                // optimiseBlockHelper(recodedHuffman(.., false))
                const SC wPP = op_recode_less(st, wY);                                    // pruned
                const SC wB2 = op_pass(st, wPP, OP_REPLACE);                              // optimiseBlockCopyHelper(pruned)
                bool full = false;
                SC wB3 = recoded_full(st, wPP, &full);                                    // prunedFull
                if (wB3.ok) {
                    nb = full ? 4 : 3;
                    if (full) wB3 = op_pass(st, wB3, OP_REPLACE);
                    trial_base(st, wB0); trial_base(st, wB1); trial_base(st, wB2);
                    if (full) trial_base(st, wB3);
                } else poisoned = true;
                if (!poisoned) D4_OR_U64(&st.doneAor, 1ull << an);
                poisoned = poisoned || outerA;
            }
            if (a == 0) {
                const SC t = op_hdr(st, wX, HOP_RECODE_LESS); cb(st, t);                        // pruned header
                long long sv = 0;
                const SC o = op_optimise(st, t, &sv); cb_if_saved(st, o, sv);
                // addOptimisedRecoded(prune) (:431) re-evaluates candidates with exactly the sizes of the sweep on `post`
                // (both are copies of the same block that differ only in the header, which every base / trial discards),
                // so under the strict `<` none of them can ever be chosen: only the index advances
                if (select) candIndex += 56u * (unsigned)nb;
            }
        }
        return !poisoned;
    }

    // one item of a discovery sweep (skipped when an earlier sweep of this round completed it) or of the selection sweep
    D4_HD bool sweep_one(SymState& st, bool sel, unsigned seg, int item) {
        if (!sel && ((st.doneItem >> item) & 1)) return true;
        const bool ok = sweep_item(st, sel, seg, item);
        if (ok && !sel) D4_OR_U32(&st.doneItem, 1u << item);
        return ok;
    }
    // every item in order: one walk over the whole enumeration, whose selection is the reference's
    D4_HD bool sweep(SymState& st, bool sel, unsigned seg) {
        bool ok = true;
        for (int i = 0; i < NITEMS; i++) ok = sweep_one(st, sel, seg, i) && ok;
        return ok;
    }

    // ---- items swept apart ------------------------------------------------------------------------------------------------
    // An item of a selection sweep that runs apart selects inside its own stretch of candidates: indices from 0, best so
    // far = the value carried into the sweep (begin_item); put_item records the outcome.  join() stitches the records
    // back in ITEM order, whatever order they were swept in: first strict minimum, indices shifted by the candidates of
    // the items before.  The result equals the walk over all items in order.
    D4_HD void begin_item(long long carried) {
        bestSize = carried; restMin = 0x7fffffffffffffffll; candIndex = 0; bestIndex = 0xffffffffu; bestStored = 0; bestArg = -1;
    }
    D4_HD void put_item(ItemRec& e) const {
        e.bestSize = bestSize; e.restMin = restMin; e.sizeC1 = sizeC1; e.best = best;
        e.bestIndex = bestIndex; e.candIndex = candIndex; e.bestStored = bestStored; e.bestArg = bestArg;
    }
    // returns true when a Huffman candidate of these items became the best
    D4_HD bool join(const ItemRec* rec) {
        bool improved = false;
        unsigned base = candIndex;
        for (int k = 0; k < NITEMS; k++) {
            const ItemRec& e = rec[k];
            if (e.bestIndex != 0xffffffffu && e.bestSize < bestSize) {
                bestSize = e.bestSize; bestIndex = base + e.bestIndex; bestStored = e.bestStored; bestArg = e.bestArg; best = e.best;
                improved = !e.bestStored;
            }
            if (e.restMin < restMin) restMin = e.restMin;
            base += e.candIndex;
        }
        candIndex = base;
        sizeC1 = rec[0].sizeC1;   // only the head item sets it
        return improved;
    }
};

}  // namespace d4
