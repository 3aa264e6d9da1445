// hosttest.cu — the single-thread building blocks of the cost model (huff.cuh) compiled as HOST code.
// TEST INFRASTRUCTURE: lets the CPU-only test suite pin the exact source the kernels execute
// (Huffman tree with java.util.PriorityQueue mechanics, header RLE packing, header trials) against the
// oracle.  Never loaded by the product.
#define D4_HOST_TEST 1
#include "huff.cuh"

using namespace d4;

extern "C" {

int host_huff_tree(const uint32_t* freq, int n, int limit, uint8_t* lens) {
    if (n <= 19) { static TreeWsCL ws; return huff_tree<21, 46>(freq, n, limit, lens, ws); }
    if (n <= 30) { static TreeWs<32, 68> ws; return huff_tree<32, 68>(freq, n, limit, lens, ws); }
    static TreeWs<290, 584> ws;
    return huff_tree<290, 584>(freq, n, limit, lens, ws);
}

// flags: bits 0-7 strategy, bit 8 prune; post_op: 0 none, 1 hdr_recode, 2 hdr_recode_less, 3 hdr_optimise
long long host_header_trial(const uint8_t* lit, int nlit, const uint8_t* dist, int ndist, int flags, int post_op,
                            int32_t* pairs_out, int32_t* np_out, int32_t* cl_out, int32_t* ncl_out) {
    static Tab t;
    static Hdr h;
    static TreeWsCL ws;
    for (int i = 0; i < MAX_LL; i++) t.L[i] = i < nlit ? lit[i] : 0;
    for (int i = 0; i < MAX_D; i++) t.D[i] = i < ndist ? dist[i] : 0;
    t.nL = (uint16_t)nlit; t.nD = (uint16_t)ndist; t.type = 2;
    if (hdr_trial(t, flags, h, ws)) return -1;
    if (post_op == 1) { if (hdr_recode(h, ws)) return -1; }
    else if (post_op == 2) { if (hdr_recode_less(h, ws)) return -1; }
    else if (post_op == 3) hdr_optimise(h);
    for (int i = 0; i < h.np; i++) { pairs_out[2 * i] = pair_run(h.pairs[i]); pairs_out[2 * i + 1] = pair_sym(h.pairs[i]); }
    *np_out = h.np;
    for (int i = 0; i < 19; i++) cl_out[i] = h.CL[i];
    *ncl_out = h.ncl;
    return h.bits;
}

int host_trial_flags(int k) { return c_trial_flags[k]; }

// the compact header-code workspace (weights must add up to less than 1024)
int host_huff_tree_compact(const uint32_t* freq, int n, int limit, uint8_t* lens) {
    static TreeWsCLc ws;
    return huff_tree_ws(freq, n, limit, lens, ws);
}

// the fast header-code tree (falls back to the compact full algorithm when deeper than the limit); *fellBack tells which
int host_huff_tree_tiny(const uint32_t* freq, int n, int limit, uint8_t* lens, int* fellBack) {
    static uint16_t heap[32];
    static uint8_t parent[64];
    static TreeWsCLc slow;
    const int rc = huff_tree_tiny(freq, n, limit, lens, heap, parent);
    *fellBack = rc == 2;
    if (rc != 2) return rc;
    return huff_tree_ws(freq, n, limit, lens, slow);
}

// size-only evaluation of one rewrite strategy for both prune values (trial_sizes over the run list)
int host_trial_sizes(const uint8_t* lit, int nlit, const uint8_t* dist, int ndist, int flags, int32_t* no_prune, int32_t* prune) {
    static Tab t;
    static RunList rl;
    static uint16_t heap[32];
    static uint8_t parent[64];
    static TreeWsCLc slow;
    TreeWsTiny ws{heap, parent, &slow};    // the workspace the engine's trial threads use
    for (int i = 0; i < MAX_LL; i++) t.L[i] = i < nlit ? lit[i] : 0;
    for (int i = 0; i < MAX_D; i++) t.D[i] = i < ndist ? dist[i] : 0;
    t.nL = (uint16_t)nlit; t.nD = (uint16_t)ndist; t.type = 2;
    runlist_build(t, rl);
    int a = 0, b = 0;
    if (trial_sizes(rl, flags, &a, &b, ws)) return 1;
    *no_prune = a; *prune = b;
    return 0;
}

}  // extern "C"

// =====================================================================================================================
// The symbolic enumerator (enum.cuh) driven by a plain serial executor: the CPU-only suite pins the very enumeration,
// memo / request / sweep logic the engine kernel runs against the oracle's candidate trace.  The executor below is the
// obvious serial statement of every request kind; the kernels' parallel versions are checked against the oracle on the
// GPU (tests/test_gpu_parity.py).
// =====================================================================================================================
#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "enum.cuh"

namespace {

struct HostEngine {
    std::vector<uint32_t> sym, symout;
    std::vector<uint8_t> out;
    uint32_t n = 0;
    uint64_t ulen = 0;
    std::vector<std::vector<uint8_t>> masks;            // one byte per symbol
    std::vector<std::array<uint32_t, 320>> hists;
    std::vector<Tab> tabs;
    std::vector<Hdr> hdrs;
    std::vector<int> trialAll;
    SymState S;
    Enumer en;
    TraceSink sink;
    unsigned traceN = 0;
    // records of B and of the winner
    Tab recTab[2]; Hdr recHdr[2]; long long recPay[2]; std::vector<uint8_t> recMask[2];
    int err = 0;
    int nSweeps = 0, nSegmented = 0, nSlowTrees = 0;

    std::array<uint32_t, 320> hist_of(const std::vector<uint8_t>& m) const {
        std::array<uint32_t, 320> h{};
        for (uint32_t i = 0; i < n; i++) {
            const uint32_t s = sym[i];
            if (!sym_is_match(s)) { if (s <= 256) h[s]++; }
            else if (!m[i]) { h[sym_lensym(s)]++; h[288 + dist_sym(sym_dist(s))]++; }
            else for (int k = 0; k < sym_len(s); k++) h[out[symout[i] + k]]++;
        }
        return h;
    }
    static long long payload_of(const std::array<uint32_t, 320>& h, const Tab& t) {
        long long acc = 0;
        for (int k = 0; k < 318; k++) {
            if (!h[k]) continue;
            int bits = 0;
            if (k < 257) bits = t.L[k];
            else if (k < 286) bits = t.L[k] + len_ebits_of(k);
            else if (k >= 288) bits = t.D[k - 288] + dist_ebits_of(k - 288);
            acc += (long long)h[k] * bits;
        }
        return acc;
    }
    int intern_mask(const std::vector<uint8_t>& m) {
        for (size_t k = 0; k < masks.size(); k++) if (masks[k] == m) return (int)k;
        if ((int)masks.size() >= MAXM) { S.overflow = 1; return 0; }
        masks.push_back(m);
        hists.push_back(hist_of(m));
        S.rc[masks.size() - 1].state = ST_EMPTY;
        S.nMasks = (int)masks.size();
        return (int)masks.size() - 1;
    }
    int intern_tab(const Tab& t) {
        for (size_t k = 0; k < tabs.size(); k++) if (!memcmp(&tabs[k], &t, sizeof(Tab))) return (int)k;
        if ((int)tabs.size() >= MAXT) { S.overflow = 1; return 0; }
        tabs.push_back(t);
        S.trialState[tabs.size() - 1] = ST_EMPTY;
        S.nTabs = (int)tabs.size();
        return (int)tabs.size() - 1;
    }
    int new_hdr(const Hdr& h) {
        if ((int)hdrs.size() >= MAXH) { S.overflow = 1; return 0; }
        hdrs.push_back(h);
        const int id = (int)hdrs.size() - 1;
        S.hbits[id] = (unsigned short)h.bits;
        S.hop[id][0] = S.hop[id][1] = S.hop[id][2] = 0;
        S.nHdrs = (int)hdrs.size();
        return id;
    }
    // literal cost - match cost of match i under t; blocked when a byte has no code
    bool dc_of(const Tab& t, uint32_t i, int* x) const {
        const uint32_t s = sym[i];
        int lit = 0;
        for (int k = 0; k < sym_len(s); k++) { const int c = t.L[out[symout[i] + k]]; if (c < 1) return false; lit += c; }
        const int ls = sym_lensym(s), ds = dist_sym(sym_dist(s));
        *x = lit - (t.L[ls] + len_ebits_of(ls) + t.D[ds] + dist_ebits_of(ds));
        return true;
    }
    void reset_pools() {
        sym_reset(S, 0, 1);
        masks.clear(); hists.clear(); tabs.clear(); hdrs.clear();
        Tab f;
        memset(&f, 0, sizeof f);
        for (int k = 0; k < 286; k++) f.L[k] = (k <= 143) ? 8 : (k <= 255) ? 9 : (k <= 279) ? 7 : 8;
        for (int k = 0; k < 30; k++) f.D[k] = 5;
        f.nL = 286; f.nD = 30; f.type = 1;
        intern_tab(f);
    }
    void adopt_B(bool toFixed) {   // from record 0
        reset_pools();
        const int mid = intern_mask(recMask[0]);
        SC b;
        b.mid = (short)mid; b.ok = 1; b.hid = -1; b.tabid = TAB_FIXED; b.type = 1; b.payload = recPay[0];
        if (toFixed) b.payload = payload_of(hists[mid], tabs[TAB_FIXED]);
        else if (recTab[0].type == 2) { b.tabid = (short)intern_tab(recTab[0]); b.hid = (short)new_hdr(recHdr[0]); b.type = 2; }
        en.B = b; en.blockType = b.type;
    }
    // instrumentation: how close is a table that needs a cost array to one that already has one?
    std::vector<int> dcSeen;
    long long statBuilds = 0, statChanged = 0, statTouched = 0, statMatches = 0, statFlip = 0, statBytesTouched = 0;
    void note_dc(int tabid) {
        for (int t : dcSeen) if (t == tabid) return;
        if (!dcSeen.empty()) {
            int best = -1, bestD = 1 << 30;
            for (int t : dcSeen) {
                int dd = 0;
                for (int b = 0; b < 256; b++) dd += tabs[t].L[b] != tabs[tabid].L[b];
                if (dd < bestD) { bestD = dd; best = t; }
            }
            bool ch[256]; bool flip = false;
            for (int b = 0; b < 256; b++) { ch[b] = tabs[best].L[b] != tabs[tabid].L[b]; if (ch[b] && (tabs[best].L[b] == 0 || tabs[tabid].L[b] == 0)) flip = true; }
            long long touched = 0, nm = 0, bt = 0;
            for (uint32_t i = 0; i < n; i++) {
                if (!sym_is_match(sym[i])) continue;
                nm++;
                int c = 0;
                for (int k = 0; k < sym_len(sym[i]); k++) c += ch[out[symout[i] + k]];
                touched += c > 0; bt += c;
            }
            { int cl = 0, cd = 0; for (int k = 257; k < 286; k++) cl += tabs[best].L[k] != tabs[tabid].L[k]; for (int k = 0; k < 30; k++) cd += tabs[best].D[k] != tabs[tabid].D[k];
              fprintf(stderr, "  dc tab %d vs %d: lit %d lensym %d dist %d touched %lld/%lld bytes %lld flip %d\n", tabid, best, bestD, cl, cd, touched, nm, bt, (int)flip); }
            statBuilds++; statChanged += bestD; statTouched += touched; statMatches += nm; statFlip += flip; statBytesTouched += bt;
        }
        dcSeen.push_back(tabid);
    }
    void exec_pass(int slot) {
        PSlot& p = S.pm[slot];
        const int mid = pm_key_mid(p.key), tabid = pm_key_tab(p.key), op = pm_key_op(p.key);
        if (op != OP_FIXED) note_dc(tabid);
        if (op == OP_FIXED) { p.delta = payload_of(hists[mid], tabs[TAB_FIXED]); p.mid = (unsigned short)mid; p.state = ST_DONE; return; }
        if ((int)masks.size() >= MAXM) { S.overflow = 1; return; }
        const Tab& t = tabs[tabid];
        std::vector<uint8_t> m = masks[mid];
        long long delta = 0;
        if (op <= OP_REPLACE_PRUNE) {
            for (uint32_t i = 0; i < n; i++) {
                if (!sym_is_match(sym[i]) || m[i]) continue;
                int x;
                if (!dc_of(t, i, &x)) continue;
                if (op == OP_REPLACE_PRUNE ? x <= 0 : x < 0) { m[i] = 1; delta -= x; }
            }
        } else {
            long long sum[32] = {0}; int cnt[32] = {0}; bool blocked[32] = {false}, seen[32] = {false};
            for (uint32_t i = 0; i < n; i++) {
                if (!sym_is_match(sym[i]) || m[i]) continue;
                const int bin = sym_lensym(sym[i]) - 257;
                seen[bin] = true;
                int x;
                if (!dc_of(t, i, &x)) { blocked[bin] = true; continue; }
                sum[bin] += x; cnt[bin]++;
            }
            int rem = -1; long long remSize = 0; int remFreq = 0;
            for (int i = 0; i < 32; i++) {
                if (blocked[i] || !seen[i]) continue;
                const bool doRem = op == OP_LEAST1 ? cnt[i] < remFreq : sum[i] < remSize;
                if (rem == -1 || doRem) { rem = i; remSize = sum[i]; remFreq = cnt[i]; }
            }
            if (rem >= 0)
                for (uint32_t i = 0; i < n; i++)
                    if (sym_is_match(sym[i]) && sym_lensym(sym[i]) - 257 == rem) m[i] = 1;
            delta = -remSize;
        }
        const int nm = intern_mask(m);
        if (S.overflow) return;
        p.mid = (unsigned short)nm; p.delta = delta; p.state = ST_DONE;
    }
    void exec_recode(int mid) {
        std::array<uint32_t, 320> h = hists[mid];
        Tab T;
        memset(&T, 0, sizeof T);
        const uint32_t* df = h.data() + 288;
        int nd = 30;
        while (nd > 0 && df[nd - 1] == 0) nd--;
        int nz = 0;
        for (int k = 0; k < nd; k++) nz += df[k] != 0;
        if (nd == 0) T.nD = 1;
        else if (nz <= 1) { T.nD = (uint16_t)nd; T.D[nd - 1] = 1; }
        else { T.nD = (uint16_t)nd; static TreeWs<32, 68> wd; if (huff_tree<32, 68>(df, nd, 15, T.D, wd)) err = 11; }
        int nl = 286;
        while (nl > 0 && h[nl - 1] == 0) nl--;
        T.nL = (uint16_t)nl;
        {   // the device's fast path, with its fallback
            std::array<uint32_t, 320> f = h;
            static uint32_t heap[296]; static uint16_t value[296];
            int rc = (ulen + n + 4 >= (1ull << 22)) ? 2 : huff_tree_fast(f.data(), nl, 15, T.L, heap, value);
            if (rc == 2) {
                nSlowTrees++;
                for (int k = 0; k < nl; k++) T.L[k] = 0;
                static TreeWs<290, 584> wl;
                if (huff_tree<290, 584>(h.data(), nl, 15, T.L, wl)) err = 11;
            }
        }
        T.type = 2;
        Hdr hd;
        memset(&hd, 0, sizeof hd);
        static TreeWsCL ws;
        if (hdr_rewrite(T, FLAGS_DEFAULT, hd, ws)) err = 11;
        const int hid = new_hdr(hd);
        const int t = intern_tab(T);
        if (S.overflow) return;
        RSlot& r = S.rc[mid];
        r.tabid = (unsigned short)t; r.hid = (unsigned short)hid; r.payload = payload_of(h, T); r.state = ST_DONE;
    }
    void exec_hdr(int q) {
        const int src = q >> 2, op = q & 3;
        Hdr h = hdrs[src];
        static TreeWsCL ws;
        if (op == HOP_RECODE) { if (hdr_recode(h, ws)) err = 11; }
        else if (op == HOP_RECODE_LESS) { if (hdr_recode_less(h, ws)) err = 11; }
        else hdr_optimise(h);
        const int id = new_hdr(h);
        if (S.overflow) return;
        S.hop[src][op] = (unsigned short)(id + 1);
    }
    void exec_trial(int t) {
        static RunList rl;
        static uint16_t heap[32];
        static uint8_t parent[64];
        static TreeWsCLc slow;
        TreeWsTiny ws{heap, parent, &slow};
        runlist_build(tabs[t], rl);
        if ((int)trialAll.size() < MAXT * 56) trialAll.assign(MAXT * 56, 0);
        for (int c = 0; c < 28; c++) {
            const int kF = c < 20 ? c : 40 + (c - 20), kT = c < 20 ? 20 + c : 48 + (c - 20);
            int a = 0, b = 0;
            if (trial_sizes(rl, c_trial_flags[kF], &a, &b, ws)) err = 11;
            trialAll[t * 56 + kF] = a; trialAll[t * 56 + kT] = b;
        }
        int best = 0x7fffffff, arg = 0;
        for (int k = 0; k < 56; k++) if (trialAll[t * 56 + k] < best) { best = trialAll[t * 56 + k]; arg = k; }
        S.trialBits[t] = (unsigned short)best; S.trialArg[t] = (unsigned char)arg; S.trialState[t] = ST_DONE;
        en.trialAll = trialAll.data();
    }
    // the PENDING entries of the memo tables -> this step's request lists (the kernel does the same with all threads).
    // Passes go in key order: which slot a pass request holds depends on which sweeper claimed it first, and its key does
    // not, so the ids the executor hands out (and with them the next sweeps) do not depend on the order of the items.
    std::vector<unsigned long long> reqLog;   // per execute level: a marker, then the sorted keys of its requests
    void collect() {
        S.nqPass = S.nqRec = S.nqHdr = S.nqTrial = 0;
        std::vector<std::pair<unsigned, int>> pend;
        for (int k = 0; k < PMEMO; k++)
            if (S.pm[k].key != 0 && S.pm[k].state != ST_DONE) pend.push_back({S.pm[k].key, k});
        std::sort(pend.begin(), pend.end());
        for (const auto& q : pend) if (S.nqPass < QPASS) S.qPass[S.nqPass++] = (unsigned short)q.second;
        for (int k = 0; k < S.nMasks; k++)
            if (S.rc[k].state == ST_PENDING && S.nqRec < QREC) S.qRec[S.nqRec++] = (unsigned short)k;
        for (int k = 0; k < S.nHdrs * 3; k++)
            if (S.hop[k / 3][k % 3] == 0xFFFF && S.nqHdr < QHDR) S.qHdr[S.nqHdr++] = (unsigned short)(((k / 3) << 2) | (k % 3));
        for (int k = 0; k < S.nTabs; k++)
            if (S.trialState[k] == ST_PENDING && S.nqTrial < QTRIAL) S.qTrial[S.nqTrial++] = (unsigned short)k;
        reqLog.push_back(~0ull);
        for (const auto& q : pend) reqLog.push_back(q.first);
        for (int k = 0; k < S.nqRec; k++) reqLog.push_back(1ull << 32 | S.qRec[k]);
        for (int k = 0; k < S.nqHdr; k++) reqLog.push_back(2ull << 32 | S.qHdr[k]);
        for (int k = 0; k < S.nqTrial; k++) reqLog.push_back(3ull << 32 | S.qTrial[k]);
    }
    void execute() {
        for (int q = 0; q < S.nqPass; q++) exec_pass(S.qPass[q]);
        for (int q = 0; q < S.nqRec; q++) exec_recode(S.qRec[q]);
        for (int q = 0; q < S.nqHdr; q++) exec_hdr(S.qHdr[q]);
        const bool others = S.nqPass + S.nqRec + S.nqHdr > 0;
        const bool doTrials = S.nqTrial && (!others || S.nqTrial >= 16);
        if (doTrials) for (int q = 0; q < S.nqTrial; q++) exec_trial(S.qTrial[q]);
    }
    void materialise(const SC& c, int arg, int which) {
        recMask[which] = masks[c.mid];
        recTab[which] = tabs[c.tabid];
        recPay[which] = c.payload;
        memset(&recHdr[which], 0, sizeof(Hdr));
        if (c.type == 2) {
            if (arg >= 0) { static TreeWsCL ws; if (hdr_trial(recTab[which], c_trial_flags[arg], recHdr[which], ws)) err = 11; }
            else recHdr[which] = hdrs[c.hid];
        }
    }
    bool segImproved = false, segmentedRound = false;
    // Order in which the items of a sweep are taken: ORDER_WALK walks them in item order with one enumerator (the
    // reference's walk; also what a traced selection does); the others sweep every item apart, as the kernel's sweepers
    // do, and join the selection records in item order.
    enum { ORDER_WALK = -1, ORDER_FORWARD = 0, ORDER_REVERSE = 1, ORDER_SHUFFLE = 2 };
    int order = ORDER_FORWARD;
    unsigned long long shuffleState = 0;
    std::vector<int> item_order() {
        std::vector<int> o(NITEMS);
        for (int i = 0; i < NITEMS; i++) o[i] = order == ORDER_REVERSE ? NITEMS - 1 - i : i;
        if (order == ORDER_SHUFFLE)
            for (int i = NITEMS - 1; i > 0; i--) {   // Fisher-Yates over a 64-bit LCG: a new permutation every sweep
                shuffleState = shuffleState * 6364136223846793005ull + 1442695040888963407ull;
                std::swap(o[i], o[(int)((shuffleState >> 33) % (unsigned long long)(i + 1))]);
            }
        return o;
    }
    bool sweep_apart(bool sel, unsigned seg) {
        bool ok = true;
        ItemRec rec[NITEMS];
        const long long carried = en.bestSize;
        for (int item : item_order()) {
            Enumer w = en;
            w.trace = nullptr;
            if (sel) w.begin_item(carried);
            ok = w.sweep_one(S, sel, seg, item) && ok;
            if (w.internalError) en.internalError = w.internalError;
            if (sel) w.put_item(rec[item]);
        }
        if (sel) segImproved = en.join(rec);
        return ok;
    }
    bool run_segment(unsigned seg) {
        S.doneItem = 0; S.doneAor = 0;
        const bool walk = order == ORDER_WALK;
        for (int it = 0;; it++) {
            nSweeps++;
            const bool done = walk ? en.sweep(S, false, seg) : sweep_apart(false, seg);
            if (S.overflow) return false;
            collect();
            const bool nothing = S.nqPass + S.nqRec + S.nqHdr + S.nqTrial == 0;
            if (done && nothing) break;
            if (nothing || it > 4096 || en.internalError) { err = 16; return false; }
            execute();
            if (S.overflow) return false;
        }
        if (walk || en.trace) {
            const unsigned before = en.bestIndex;
            if (!en.sweep(S, true, seg)) err = 16;
            segImproved = en.bestIndex != before && !en.bestStored;
        } else if (!sweep_apart(true, seg)) err = 16;
        if (en.internalError) err = 16;
        return true;
    }
    void optimise_block(long long storedSize, bool forceSegmented) {
        en.storedSize = storedSize;
        en.begin_round(S);
        segmentedRound = false;
        bool ok = !forceSegmented && run_segment(Enumer::SEG_ALL);
        if (ok) { materialise(en.best, en.bestArg, 1); return; }
        if (err) return;
        nSegmented++;
        segmentedRound = true;   // the winner's ids belong to pools that are gone
        materialise(en.B, -1, 0);
        en.begin_round(S);
        const unsigned segs[4] = {Enumer::SEG_HEAD | Enumer::SEG_MULTI_H, Enumer::SEG_MULTI_O, Enumer::SEG_FIXED | Enumer::SEG_LEAST0, Enumer::SEG_LEAST1};
        bool haveBest = false;
        for (int k = 0; k < 4; k++) {
            const long long bs = en.bestSize, rm = en.restMin, c1 = en.sizeC1;
            const unsigned bi = en.bestIndex, ci = en.candIndex;
            const int bst = en.bestStored;
            adopt_B(false);
            en.bestSize = bs; en.bestIndex = bi; en.candIndex = ci; en.bestStored = bst; en.restMin = rm; en.sizeC1 = c1;
            if (!run_segment(segs[k])) { if (!err) err = 15; break; }
            if (segImproved) { materialise(en.best, en.bestArg, 1); haveBest = true; }
        }
        if (!haveBest && !err) { adopt_B(false); materialise(en.B, -1, 1); }
    }
    void advance_to_best(bool keepPools) {
        recTab[0] = recTab[1]; recHdr[0] = recHdr[1]; recPay[0] = recPay[1]; recMask[0] = recMask[1];
        const bool keep = keepPools && !segmentedRound && !S.overflow && S.nMasks <= MAXM / 2 && S.nTabs <= MAXT / 2 && S.nHdrs + 1 <= MAXH / 2 &&
                          S.nP <= PMEMO * 3 / 8 && en.bestIndex != 0xffffffffu;
        if (keep) {
            SC b = en.best;
            if (b.type == 2 && en.bestArg >= 0) b.hid = (short)new_hdr(recHdr[0]);
            en.B = b; en.blockType = b.type;
        } else adopt_B(false);
    }
};

HostEngine* g_he = nullptr;

}  // namespace

extern "C" {

// Load a block: packed symbols (common.cuh), block-relative decoded offsets, decoded bytes, the parsed tables / header.
// pairs: {sym, run, val} triples.
void* host_engine_load(const uint32_t* sym, const uint32_t* symout, uint32_t n, const uint8_t* out, uint64_t ulen, int type,
                       const uint8_t* L, int nL, const uint8_t* D, int nD, const int32_t* pairs, int np, const uint8_t* CL, int ncl,
                       int hdrBits, long long payload, int toFixed) {
    HostEngine* e = new HostEngine();
    e->sym.assign(sym, sym + n); e->symout.assign(symout, symout + n); e->out.assign(out, out + ulen);
    e->n = n; e->ulen = ulen;
    memset(&e->recTab[0], 0, sizeof(Tab)); memset(&e->recHdr[0], 0, sizeof(Hdr));
    Tab& t = e->recTab[0];
    for (int i = 0; i < nL && i < MAX_LL; i++) t.L[i] = L[i];
    for (int i = 0; i < nD && i < MAX_D; i++) t.D[i] = D[i];
    t.nL = (uint16_t)nL; t.nD = (uint16_t)nD; t.type = (uint8_t)type;
    if (type == 1) { t.nL = 286; t.nD = 30; }
    Hdr& h = e->recHdr[0];
    for (int i = 0; i < np; i++) h.pairs[i] = pair_pack(pairs[3 * i], pairs[3 * i + 1], pairs[3 * i + 2]);
    h.np = (uint16_t)np;
    for (int i = 0; i < 19; i++) h.CL[i] = CL ? CL[i] : 0;
    h.ncl = (uint8_t)ncl; h.bits = hdrBits;
    e->recPay[0] = payload;
    e->recMask[0].assign(n, 0);
    e->en.trialAll = nullptr;
    e->en.trace = nullptr;
    e->en.storedOK = ulen <= 65535;
    e->adopt_B(toFixed != 0);
    return e;
}
void host_engine_free(void* p) { delete (HostEngine*)p; }

// One optimiseBlock call.  res: {bestSize, bestIndex, bestStored, sizeI, sizeC1, restMin, candIndex (total), err, sweeps,
// segmented, masks, tabs, hdrs, memo entries, slow trees, size of the materialised winner}.  trace: (index, size) pairs.
int host_engine_round(void* p, long long storedSize, int forceSegmented, long long* res, long long* trace, unsigned traceCap,
                      unsigned* traceN) {
    HostEngine* e = (HostEngine*)p;
    e->traceN = 0;
    e->sink.buf = trace; e->sink.cap = traceCap; e->sink.n = &e->traceN;
    e->en.trace = trace ? &e->sink : nullptr;
    e->nSweeps = 0; e->nSegmented = 0;
    e->optimise_block(storedSize, forceSegmented != 0);
    res[0] = e->en.bestSize; res[1] = e->en.bestIndex; res[2] = e->en.bestStored; res[3] = e->en.sizeI; res[4] = e->en.sizeC1;
    res[5] = e->en.restMin; res[6] = e->en.candIndex; res[7] = e->err; res[8] = e->nSweeps; res[9] = e->nSegmented;
    res[10] = e->S.nMasks; res[11] = e->S.nTabs; res[12] = e->S.nHdrs; res[13] = e->S.nP; res[14] = e->nSlowTrees;
    res[15] = e->recPay[1] + (e->recTab[1].type == 2 ? e->recHdr[1].bits : 0);
    if (getenv("D4_HOST_DCSTATS")) fprintf(stderr, "dcstats builds %lld avg_changed_bytes %.2f touched_frac %.3f flips %lld byte_updates_per_build %.0f matches %lld\n", e->statBuilds, e->statBuilds ? (double)e->statChanged / e->statBuilds : 0.0, e->statMatches ? (double)e->statTouched / e->statMatches : 0.0, e->statFlip, e->statBuilds ? (double)e->statBytesTouched / e->statBuilds : 0.0, e->statBuilds ? e->statMatches / e->statBuilds : 0);
    if (traceN) *traceN = e->traceN;
    return e->err;
}
// order of the items of every following sweep (HostEngine::ORDER_*); seed: the shuffle's
void host_engine_order(void* p, int order, unsigned long long seed) {
    HostEngine* e = (HostEngine*)p;
    e->order = order; e->shuffleState = seed;
}
// selection state after the last round: {bestSize, bestIndex, bestStored, bestArg, restMin, sizeC1, candIndex}
void host_engine_selection(void* p, long long* out) {
    const Enumer& en = ((HostEngine*)p)->en;
    out[0] = en.bestSize; out[1] = en.bestIndex; out[2] = en.bestStored; out[3] = en.bestArg; out[4] = en.restMin;
    out[5] = en.sizeC1; out[6] = en.candIndex;
}
// the request log since the block was loaded: per execute level ~0, then its requests (pass keys; 1 << 32 | mask id of a
// recode; 2 << 32 | hid << 2 | op of a header op; 3 << 32 | table id of a trial).  Returns its length.
size_t host_engine_reqlog(void* p, unsigned long long* buf, size_t cap) {
    const auto& l = ((HostEngine*)p)->reqLog;
    for (size_t k = 0; k < l.size() && k < cap; k++) buf[k] = l[k];
    return l.size();
}
// the winner becomes the block (the next optimiseBlock call of DeflateStream.optimise's loop)
void host_engine_advance(void* p, int keepPools) { ((HostEngine*)p)->advance_to_best(keepPools != 0); }
// the materialised winner: code lengths, header, mask (one byte per symbol)
void host_engine_best(void* p, uint8_t* L, uint8_t* D, int32_t* meta, int32_t* pairs, uint8_t* CL, uint8_t* mask) {
    HostEngine* e = (HostEngine*)p;
    const Tab& t = e->recTab[1];
    const Hdr& h = e->recHdr[1];
    memcpy(L, t.L, MAX_LL); memcpy(D, t.D, MAX_D);
    meta[0] = t.type; meta[1] = t.nL; meta[2] = t.nD; meta[3] = h.np; meta[4] = h.ncl; meta[5] = h.bits;
    for (int i = 0; i < h.np; i++) { pairs[2 * i] = pair_run(h.pairs[i]); pairs[2 * i + 1] = pair_sym(h.pairs[i]); }
    memcpy(CL, h.CL, 19);
    memcpy(mask, e->recMask[1].data(), e->n);
}

}  // extern "C"

// =====================================================================================================================
// The compressor's parse rule (lzrule.cuh) on the host: the fixed-coded stream F the device compressor models, written
// with a plain serial hash chain over the whole stream.  The GPU's F is compared with this byte for byte.
// =====================================================================================================================
#include "lzrule.cuh"

namespace {
struct HostBits {
    std::vector<uint8_t> out;
    uint64_t acc = 0;
    int n = 0;
    void bits(uint32_t v, int c) {
        acc |= (uint64_t)v << n;
        n += c;
        while (n >= 8) { out.push_back((uint8_t)acc); acc >>= 8; n -= 8; }
    }
    void code(uint32_t c, int len) {   // Huffman codes go MSB first
        uint32_t r = 0;
        for (int k = 0; k < len; k++) r |= ((c >> k) & 1u) << (len - 1 - k);
        bits(r, len);
    }
    void fixed_lit(int s) {
        if (s <= 143) code(0x30 + s, 8);
        else if (s <= 255) code(0x190 + s - 144, 9);
        else if (s <= 279) code(s - 256, 7);
        else code(0xC0 + s - 280, 8);
    }
};
struct HostByte { const uint8_t* d; __host__ __device__ uint8_t operator()(int64_t i) const { return d[i]; } };
struct HostLink { const int64_t* prev; __host__ __device__ int64_t operator()(int64_t q) const { return prev[q]; } };
}  // namespace

extern "C" {

// F for `n` bytes at block size `block`; returns its size in bits (-1: `cap` too small), bytes in out[0, ceil(bits / 8))
long long host_lz_compress(const uint8_t* d, uint64_t n, uint32_t block, uint8_t* out, uint64_t cap) {
    std::vector<int64_t> prev(n, -1), head(LZ_HASH_MASK + 1, -1);
    for (uint64_t p = 0; p + 3 <= n; p++) {
        const uint32_t h = lz_hash(d[p], d[p + 1], d[p + 2]);
        prev[p] = head[h];
        head[h] = (int64_t)p;
    }
    const HostByte byte{d};
    const HostLink link{prev.data()};
    HostBits w;
    long long bits = 0;
    const uint64_t nblk = n == 0 ? 1 : (n + block - 1) / block;
    for (uint64_t b = 0; b < nblk; b++) {
        const int64_t s = (int64_t)(b * block), e = (int64_t)std::min<uint64_t>(n, (b + 1) * block);
        w.bits(b + 1 == nblk ? 1 : 0, 1);
        w.bits(1, 2);
        bits += 3;
        std::vector<uint32_t> M(e - s + 1, 0);
        for (int64_t p = s; p < e; p++) M[p - s] = lz_best_match(p, e, (int64_t)n, byte, link);
        for (int64_t i = s; i < e;) {
            const uint32_t m = lz_take(M[i - s], M[i + 1 - s], i + 1 == e);
            if (m) {
                const int len = (int)lz_mlen(m), dist = (int)lz_mdist(m);
                const int ls = lz_len_sym(len), ds = dist_sym(dist);
                w.fixed_lit(ls);
                w.bits((uint32_t)(len - c_len_base[ls - 257]), len_ebits_of(ls));
                w.code((uint32_t)ds, 5);
                w.bits((uint32_t)(dist - c_dist_base[ds]), dist_ebits_of(ds));
                bits += lz_fixed_match_bits(len, dist);
                i += len;
            } else {
                w.fixed_lit(d[i]);
                bits += lz_fixed_lit_bits(d[i]);
                i++;
            }
        }
        w.fixed_lit(256);
        bits += LZ_FIXED_EOB_BITS;
    }
    if (w.n) w.bits(0, 8 - w.n);
    if (w.out.size() > cap) return -1;
    memcpy(out, w.out.data(), w.out.size());
    return bits;
}

}  // extern "C"
