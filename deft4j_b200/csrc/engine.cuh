// engine.cuh — the block candidate engine: executes what the symbolic enumerator (enum.cuh) asks for.
//
// One CTA owns one block.  Lane 0 of every warp sweeps items of the enumeration of DeflateStream.optimiseBlock
// (DeflateStream.java:343-490) over memo tables in shared memory; every miss becomes a request.  After a sweep the whole CTA computes the requests:
//   passes   replaceBackrefsWithLiteralsIfSmaller / removeDistLitLeastExpensive (DeflateBlockHuffman.java:222-319,
//            373-458): CTA-wide, 8 matches per thread, against a per-table cost array dc[j] = literal cost - match cost.
//            The cost array of a table is built in ONE coalesced pass over the block's decoded bytes: 2 KiB tiles, per-byte
//            code lengths looked up in shared memory, a CTA-wide prefix sum per tile, every match takes P[end] - P[start].
//   recodes  recodeHuffman (:670-743): one WARP per request - histogram row -> litlen and distance Huffman trees with the
//            exact java.util.PriorityQueue mechanics (lane 0; the trees of up to 8 requests run side by side) -> payload
//            (dot product) -> default header (runs -> pairs -> header code), all inside the warp.
//   headers  recodeHeader / recodeHeaderToLessRLEMatches / optimiseHeader (:471-476,579-635): one warp per request.
//   trials   the 56 header strategies of a table (DeflateStream.java:277-316): 28 threads per table, 8 tables at a time,
//            sizes only (huff.cuh trial_sizes); the winner alone is materialised.
// Inside the engine a block is its matches: match j is the j-th match in symbol order, and every per-block array (masks,
// cost arrays, sign masks, match records) is indexed by j, since literals never change.  The mask pool outside the engine
// keeps one bit per symbol; load_block and store_mask translate.
// Masks (symbol lists), Tabs and Hdrs are immutable entries of per-CTA pools in global scratch, hash-consed where it
// pays (masks, Tabs); a pool that fills up makes the round restart in segments with a reset between them.
#pragma once
#include "enum.cuh"
#include "parse.cuh"

namespace d4 {

#ifndef D4_ENG_NT
#define D4_ENG_NT 256
#endif
#ifndef D4_ENG_MINB
#define D4_ENG_MINB 4
#endif
constexpr int ENG_NT = D4_ENG_NT;
constexpr int ENG_NW = ENG_NT / 32;
constexpr int ERR_TREE = 11, ERR_ROUNDS = 12, ERR_WRITER = 2, ERR_POOL = 15, ERR_INTERNAL = 16;  // reported through gerr

// parity-debug instrumentation (deft4cu_debug_trace): when armed, every candidate the selection callback sees is logged
// as (candidate index, size)
__device__ long long* g_trace = nullptr;
__device__ unsigned g_trace_cap = 0;
__device__ unsigned g_trace_n = 0;

struct Cand {               // a materialised candidate (BlkState, the records of the current and the best block)
    Tab tab;
    Hdr hdr;
    long long payload;      // litlenSizeBits
    uint16_t mid, tabid;    // unused outside the engine
    uint32_t pad2;
};
__device__ __forceinline__ long long cand_size(const Cand& c) { return c.payload + (c.tab.type == 2 ? c.hdr.bits : 0); }

struct BlkView {
    const uint32_t* sym;
    const uint32_t* symout;
    const uint8_t* out;
    uint32_t n;       // symbols (including NOPs left by a merge)
    uint32_t nm;      // matches (build_views)
    uint32_t nwords;  // mask words: the engine's masks have one bit per match (build_views)
    uint64_t ulen;    // decoded length
    uint64_t out_off; // pool offset of the block's first decoded byte
};

constexpr int DC_TILE = 512;      // decoded bytes per cost-array tile: one 16-byte load per lane of a warp
// Cache and queue capacities.  Each is a macro so that a stress build can shrink it until every eviction, reset and
// overflow path runs on ordinary inputs (__graft_entry__.build: libdeft4cu_stress.so); the product build uses the defaults.
#ifndef D4_DCN
#define D4_DCN 16
#endif
#ifndef D4_LCN
#define D4_LCN 12
#endif
#ifndef D4_MAXLIT
#define D4_MAXLIT 64
#endif
#ifndef D4_HQS
#define D4_HQS 4608
#endif
#ifndef D4_HQL
#define D4_HQL 1024
#endif
constexpr int DCN = D4_DCN;       // per-table sign masks kept per block (round-robin eviction)
constexpr int LCN = D4_LCN;       // literal-cost arrays kept per block (round-robin eviction)
constexpr int MAXLIT = D4_MAXLIT; // distinct sets of literal code lengths tracked per block
constexpr int WS_BYTES = 3072;    // per-warp workspace for trees / header work
constexpr int HQS = D4_HQS, HQL = D4_HQL;   // queue of freshly replaced matches (all / long ones) for the histogram update
// a pass holds one literal-cost array and one sign-mask slot at a time; the slot indices are stored in unsigned chars
// whose 0xFF means "none"
static_assert(DCN >= 1 && DCN < 0xFF && LCN >= 1 && LCN < 0xFF && MAXLIT >= 1 && MAXLIT < 0xFF, "cache sizes");
static_assert(HQS >= 1 && HQL >= 1, "queue sizes");
constexpr int SLOT_B = MAXM, SLOT_BEST = MAXM + 1;   // extra mask / histogram slots: the records of B and of the winner
static_assert(DC_TILE == 32 * 16 && DC_TILE > 258, "a tile is one warp-wide 128-bit load and no match spans more than two tiles");

// cycle accounting per engine phase (-DD4_PROF builds only; read back with deft4cu_debug_prof): thread 0's clock64
// deltas (a sweep counts up to the barrier after it, so it is the slowest sweeper's time), [cat] = cycles, [32 + cat] = calls
#ifdef D4_PROF
__device__ unsigned long long g_prof[64];
#define P0() const long long p0_ = clock64()
#define P1(cat) do { if (threadIdx.x == 0) { atomicAdd(&g_prof[cat], (unsigned long long)(clock64() - p0_)); atomicAdd(&g_prof[32 + (cat)], 1ull); } } while (0)
#define PCOUNT(cat, k) do { if (threadIdx.x == 0) atomicAdd(&g_prof[32 + (cat)], (unsigned long long)(k)); } while (0)
#else
#define P0()
#define P1(cat)
#define PCOUNT(cat, k)
#endif
enum { PR_BLOCK = 0, PR_ROUND, PR_SWEEP, PR_SELECT, PR_PASS, PR_DC, PR_RECODE, PR_TREES, PR_HDR_DEFAULT, PR_HDROP, PR_TRIALS,
       PR_LOAD, PR_MATERIAL, PR_REBASE, PR_INTERN_MASK, PR_INTERN_TAB, PR_FIXED, PR_SLOWTREE, PR_SEGMENTED, PR_HIST,
       PR_PASS_MAIN, PR_PASS_HQ, PR_LEAST_APPLY, PR_PASS_LEAST, PR_MASKS };

struct EngSmem {
    SymState sym;
    Enumer en;            // the block, the round's selection state, and the sweeper of a traced selection sweep
    TraceSink tsink;
    unsigned long long maskHash[MAXM];
    uint32_t hist[320];          // pass histogram delta / block histogram; [0,19) header pair frequencies
    int leastSum[32], leastCnt[32];
    unsigned leastBlocked, leastSeen;
    int leastRem[2], leastSize[2];   // the length symbol each mode removes and its cost sum
    const short* hqLit;              // replace pass in progress: its literal-cost array (nullptr otherwise)
    uint32_t binStart[33];           // perm[binStart[b] .. binStart[b + 1]) = the matches with length symbol 257 + b
    uint32_t itemStart[33];          // items[itemStart[b] .. itemStart[b + 1]) cover bin b, 32 matches apiece
    unsigned long long red;
    unsigned long long hred[ENG_NW];
    long long recPay[ENG_NW];
    uint32_t wt[ENG_NW];
    int redAny, redAny2, tmpIdx, err;
    int itemNext, segImproved, segmentedRound;   // itemNext: the next item of the current sweep
    unsigned char tabDc[MAXT];   // tabid -> sign-mask slot (0xFF: none)
    unsigned short dcOwner[DCN]; // slot -> tabid (0xFFFF: free)
    int dcNext;
    // literal-cost arrays are shared by all tables with the same literal code lengths
    unsigned char tabLit[MAXT];          // tabid -> literal set (0xFF: not looked up yet)
    unsigned long long litHash[MAXLIT];  // literal set -> hash of its 256 code lengths
    unsigned short litRep[MAXLIT];       // ... a table that has it
    unsigned char litSlot[MAXLIT];       // ... its cost-array slot (0xFF: none)
    unsigned char slotLit[LCN];          // slot -> literal set (0xFF: free)
    int nLit, litNext;
    uint32_t ctab[256];          // cost-array build: literal code lengths (0x10000 = no code: counted apart)
    uint8_t refL[32], refD[32];  // cost of a match's length symbol / distance symbol incl. extra bits
    union alignas(16) {
        unsigned char ws[ENG_NW][WS_BYTES];
        uint32_t P[ENG_NW][DC_TILE + 4 + 36]; // cost-array build: per warp, packed (cost | uncodable count << 16) prefixes of one tile + lane bases
        struct { Tab tab; Hdr hdr; TreeWsCL ws; } mat;   // winner materialisation (thread 0)
        struct { Enumer w[ENG_NW]; ItemRec rec[NITEMS]; } sw;   // sweeps: the sweepers' enumerators, the selection of every item
        struct { uint32_t nS, nL; uint32_t qs[HQS]; uint32_t ql[HQL]; } hq;   // passes: matches that were just replaced
    } u;
};

// Global scratch: ONE contiguous slab per CTA (2 MiB aligned) holding all of its pools and views, so that a CTA's working
// set sits in a handful of pages (twelve separate arrays indexed by CTA cost a TLB miss on almost every access).
// The engine state of the CTA.  A file-scope __shared__ object (every kernel that uses the engine gets its own copy), so
// that the compiler knows the address space of every access (LDS / STS / ATOMS instead of generic LD / ST / ATOM).
__shared__ EngSmem g_es;
#define ES (&g_es)

struct EngScratch {
    unsigned char* slab;
    size_t stride;        // bytes per CTA
    // byte offsets inside a CTA's slab
    size_t oMasks;        // (MAXM + 2) * maxwords u32 (slot SLOT_BEST doubles as a symbol-space mask in k_finish)
    size_t oTabs;         // MAXT + ENG_NW (staging) Tab
    size_t oHdrs;         // MAXH Hdr
    size_t oHists;        // (MAXM + 2) * 320 u32
    size_t oTabHash;      // MAXT u64
    size_t oDc;           // LCN * maxwords * 32 short: literal-cost arrays
    size_t oMinfo;        // maxwords * 32 u32: per match, its packed record (build_views)
    size_t oMout;         // maxwords * 32 u32: per match, the pool offset of its first decoded byte
    size_t oMflag;        // maxwords u32: per symbol word, which of its symbols are matches
    size_t oMrank;        // maxwords u32: per symbol word, the matches before its first symbol
    size_t oLitHist;      // 320 u32: histogram of the block's literals and EOB
    size_t oTileFirst;    // maxtiles u32
    size_t oTrialAll;     // MAXT * 56 int
    size_t oRecs;         // 2 Cand: B and the winner
    size_t oSlowWs;       // ENG_NW TreeWs<290, 584>
    size_t oPerm;         // maxwords * 32 u32: the block's match ranks grouped by length symbol
    size_t oDcBits;       // DCN * 2 * maxwords u32: per cost array, the matches with a negative / a zero entry
    size_t oItems;        // maxwords + 64 u32: stretches of <= 32 entries of perm with one length symbol
    uint32_t maxwords, maxtiles;
};
// lays the slab out; returns the stride.  maxwords bounds the symbol words of a block, so it bounds its match words too.
inline size_t eng_scratch_layout(EngScratch& sc, uint32_t maxwords, uint64_t maxu) {
    sc.maxwords = maxwords;
    sc.maxtiles = (uint32_t)(maxu / DC_TILE + 4);
    const size_t maxn = (size_t)maxwords * 32;
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = (o + bytes + 255) & ~(size_t)255; return at; };
    // the small, hot arrays first
    sc.oRecs = take(2 * sizeof(Cand));
    sc.oTabHash = take(sizeof(unsigned long long) * MAXT);
    sc.oTabs = take(sizeof(Tab) * (MAXT + ENG_NW));
    sc.oLitHist = take(4 * 320);
    sc.oMflag = take(4 * (size_t)maxwords);
    sc.oMrank = take(4 * (size_t)maxwords);
    sc.oTileFirst = take(4 * (size_t)sc.maxtiles);
    sc.oMinfo = take(4 * maxn);
    sc.oMout = take(4 * maxn);
    sc.oPerm = take(4 * maxn);
    sc.oItems = take(4 * ((size_t)maxwords + 64));
    sc.oDc = take(2 * maxn * LCN);
    sc.oDcBits = take(4 * (size_t)maxwords * 2 * DCN);
    sc.oMasks = take(4 * (size_t)(MAXM + 2) * maxwords);
    sc.oHists = take(4 * (size_t)(MAXM + 2) * 320);
    sc.oHdrs = take(sizeof(Hdr) * MAXH);
    sc.oTrialAll = take(4 * (size_t)MAXT * 56);
    sc.oSlowWs = take(sizeof(TreeWs<290, 584>) * ENG_NW);
    sc.stride = (o + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1);
    return sc.stride;
}

struct Eng {
    // cost-array value that is not a cost: a match with a byte that has no code
    static constexpr short DC_BLOCKED = 0x7FFF;
    BlkView v;
    uint32_t* masks;
    uint32_t maxwords, maxn;
    Tab* tabs;
    Hdr* hdrs;
    uint32_t* hists;
    unsigned long long* tabHash;
    short* dc;            // literal-cost arrays (LCN slots of maxn)
    uint32_t* minfo;      // per match: len-3 | dist symbol << 9 | (length symbol - 256) << 14 | (start in its cost tile) << 19
    uint32_t* mout;       // per match: pool offset of its first decoded byte
    uint32_t* mflag;      // per symbol word: bit b = symbol 32k + b is a match
    uint32_t* mrank;      // per symbol word: rank of its first match
    uint32_t* litHist;    // the block's literals and EOB: the part of every histogram that no pass changes
    uint32_t* tileFirst;  // per cost tile: the first match that starts in it or later
    int* trialAll;
    Cand* recs;
    TreeWs<290, 584>* slowWs;
    uint32_t* perm;       // ranks of the block's matches, grouped by length symbol (ES->binStart)
    uint32_t* dcBits;     // per cost array: maxwords words 'entry < 0', then maxwords words 'entry == 0'
    uint32_t* items;      // work items of the least-expensive statistics: first perm index | length symbol bin << 27
    int tid;
    bool bigWeights;     // the histogram total may not fit the fast tree's 22-bit weights

    __device__ uint32_t* maskp(int id) const { return masks + (size_t)id * maxwords; }
    __device__ uint32_t* histp(int id) const { return hists + (size_t)id * 320; }

    __device__ __noinline__ unsigned long long hash_words(const uint32_t* p, int nwords32) {
        unsigned long long h = 0;
#pragma unroll 1
        for (int k = tid; k < nwords32; k += ENG_NT) {
            unsigned long long x = (unsigned long long)p[k] + 0x9E3779B97F4A7C15ull * (unsigned long long)(k + 1);
            x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
            h += x;
        }
#pragma unroll 1
        for (int d = 16; d > 0; d >>= 1) h += __shfl_xor_sync(0xffffffffu, h, d);
        if ((tid & 31) == 0) ES->hred[tid >> 5] = h;
        __syncthreads();
        unsigned long long r = 0;
#pragma unroll 1
        for (int k = 0; k < ENG_NW; k++) r += ES->hred[k];
        __syncthreads();
        return r | 1ull;
    }
    static __device__ __forceinline__ unsigned long long hash_words_warp(const uint32_t* p, int nwords32, int lane) {
        unsigned long long h = 0;
#pragma unroll 1
        for (int k = lane; k < nwords32; k += 32) {
            unsigned long long x = (unsigned long long)p[k] + 0x9E3779B97F4A7C15ull * (unsigned long long)(k + 1);
            x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
            h += x;
        }
#pragma unroll 1
        for (int d = 16; d > 0; d >>= 1) h += __shfl_xor_sync(0xffffffffu, h, d);
        return h | 1ull;
    }

    // ---- pools ----------------------------------------------------------------------------------------------------
    // the Tab in staging slot `st` -> its id (hash-consed; a hash hit is confirmed by a full comparison).  One warp.
    __device__ __noinline__ int intern_tab_warp(int st, int lane) {
        const uint32_t* q = (const uint32_t*)&tabs[MAXT + st];
        const unsigned long long h = hash_words_warp(q, (int)(sizeof(Tab) / 4), lane);
        const int nT = ES->sym.nTabs;
        int hit = -1;
#pragma unroll 1
        for (int k0 = 0; k0 < nT && hit < 0; k0 += 32) {
            const int k = k0 + lane;
            unsigned m = __ballot_sync(0xffffffffu, k < nT && tabHash[k] == h);
            while (m && hit < 0) {
                const int cand = k0 + __ffs((int)m) - 1;
                m &= m - 1;
                const uint32_t* a = (const uint32_t*)&tabs[cand];
                bool diff = false;
#pragma unroll 1
                for (int w = lane; w < (int)(sizeof(Tab) / 4); w += 32) diff |= a[w] != q[w];
                if (!__any_sync(0xffffffffu, diff)) hit = cand;
            }
        }
        if (hit < 0) {
            if (nT >= MAXT) { if (lane == 0) ES->sym.overflow = 1; return 0; }
            hit = nT;
            uint32_t* a = (uint32_t*)&tabs[hit];
#pragma unroll 1
            for (int w = lane; w < (int)(sizeof(Tab) / 4); w += 32) a[w] = q[w];
            if (lane == 0) { tabHash[hit] = h; ES->sym.trialState[hit] = ST_EMPTY; ES->sym.nTabs = nT + 1; }
            __syncwarp();
        }
        return hit;
    }

    // Mask hash = sum over the non-zero mask bytes of a mix of (byte, byte index): the passes accumulate it while they
    // write the mask, so interning needs no extra walk.
    static __device__ __forceinline__ unsigned long long mask_byte_hash(uint32_t byteval, uint32_t byteidx) {
        if (!byteval) return 0ull;
        unsigned long long x = (unsigned long long)byteval | ((unsigned long long)byteidx << 8);
        x *= 0x9E3779B97F4A7C15ull; x ^= x >> 29; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 32;
        return x;
    }
    __device__ __noinline__ unsigned long long cta_sum64(unsigned long long h) {
#pragma unroll 1
        for (int d = 16; d > 0; d >>= 1) h += __shfl_xor_sync(0xffffffffu, h, d);
        __syncthreads();
        if ((tid & 31) == 0) ES->hred[tid >> 5] = h;
        __syncthreads();
        unsigned long long r = 0;
#pragma unroll 1
        for (int k = 0; k < ENG_NW; k++) r += ES->hred[k];
        return r;
    }
    __device__ __noinline__ unsigned long long mask_hash_cta(const uint32_t* m) {
        unsigned long long h = 0;
#pragma unroll 1
        for (uint32_t k = tid; k < v.nwords; k += ENG_NT) {
            const uint32_t w = m[k];
            if (!w) continue;
#pragma unroll
            for (int q = 0; q < 4; q++) h += mask_byte_hash((w >> (8 * q)) & 0xffu, 4 * k + q);
        }
        return cta_sum64(h);
    }

    // the mask just written into pool slot nMasks (hash h) -> its id (an equal older mask wins, so equal symbol lists
    // reached along different paths share their memo entries)
    __device__ __noinline__ int intern_mask(unsigned long long h) {
        P0();
        const int fresh = ES->sym.nMasks;
        const uint32_t* q = maskp(fresh);
        __syncthreads();
        if (tid == 0) { ES->tmpIdx = -1; ES->redAny2 = 0; }
        __syncthreads();
#pragma unroll 1
        for (int k = tid; k < fresh; k += ENG_NT)
            if (ES->maskHash[k] == h) atomicMax(&ES->tmpIdx, k);
        __syncthreads();
        int hit = ES->tmpIdx;
        if (hit >= 0) {
            const uint32_t* a = maskp(hit);
            bool diff = false;
#pragma unroll 1
            for (uint32_t k = tid; k < v.nwords; k += ENG_NT) diff |= a[k] != q[k];
            if (diff) ES->redAny2 = 1;
            __syncthreads();
            if (ES->redAny2) hit = -1;
        }
        __syncthreads();
        if (hit < 0) {
            hit = fresh;
            if (tid == 0) { ES->maskHash[fresh] = h; ES->sym.rc[fresh].state = ST_EMPTY; ES->sym.nMasks = fresh + 1; }
        }
        __syncthreads();
        P1(PR_INTERN_MASK);
        return hit;
    }

    // ---- block load -----------------------------------------------------------------------------------------------
    __device__ __forceinline__ uint32_t sym_words() const { return (v.n + 31) / 32; }

    // The views the passes read, all indexed by match rank j: minfo[j] (see its declaration), mout[j], perm (the ranks
    // grouped by length symbol) and tileFirst[t] = first match that starts in tile t or later (tiles count from the
    // 16-byte boundary at or below the block's first decoded byte); mflag / mrank translate symbol words to ranks;
    // litHist = the histogram of the literals and the EOB.  Sets v.nm and v.nwords.
    __device__ __noinline__ void build_views() {
        const int lane = tid & 31, wid = tid >> 5;
        const uint32_t nsw = sym_words();
#pragma unroll 1
        for (uint32_t k = (uint32_t)wid; k < nsw; k += ENG_NW) {
            const uint32_t i = 32 * k + (uint32_t)lane;
            const uint32_t f = __ballot_sync(0xffffffffu, i < v.n && sym_is_match(v.sym[i]));
            if (lane == 0) mflag[k] = f;
        }
#pragma unroll 1
        for (int k = tid; k < 320; k += ENG_NT) ES->hist[k] = 0;
        if (tid < 32) ES->leastCnt[tid] = 0;
        __syncthreads();
        // ranks: every thread owns a contiguous run of symbol words, CTA-wide exclusive scan of their match counts
        {
            const uint32_t per = (nsw + ENG_NT - 1) / ENG_NT;
            const uint32_t k0 = min(nsw, (uint32_t)tid * per), k1 = min(nsw, k0 + per);
            uint32_t c = 0;
#pragma unroll 1
            for (uint32_t k = k0; k < k1; k++) c += (uint32_t)__popc(mflag[k]);
            uint32_t incl = c;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, incl, dd); if (lane >= dd) incl += y; }
            if (lane == 31) ES->wt[wid] = incl;
            __syncthreads();
            uint32_t base = incl - c, total = 0;
#pragma unroll 1
            for (int w = 0; w < ENG_NW; w++) { const uint32_t x = ES->wt[w]; if (w < wid) base += x; total += x; }
#pragma unroll 1
            for (uint32_t k = k0; k < k1; k++) { mrank[k] = base; base += (uint32_t)__popc(mflag[k]); }
            v.nm = total;
            v.nwords = (total + 31) / 32;
        }
        __syncthreads();
        // match records; literals and EOB into the fixed histogram
        const uint32_t a0 = (uint32_t)(v.out_off & ~15ull);
#pragma unroll 1
        for (uint32_t k = (uint32_t)wid; k < nsw; k += ENG_NW) {
            const uint32_t i = 32 * k + (uint32_t)lane;
            if (i >= v.n) continue;
            const uint32_t f = mflag[k];
            const uint32_t s = v.sym[i];
            if ((f >> lane) & 1) {
                const uint32_t j = mrank[k] + (uint32_t)__popc(f & ((1u << lane) - 1u));
                const uint32_t so = v.symout[i];
                const uint32_t kq = (uint32_t)(sym_lensym(s) - 256), dsy = (uint32_t)dist_sym(sym_dist(s));
                minfo[j] = (s & 0x1FF) | (dsy << 9) | (kq << 14) | (((so - a0) & (DC_TILE - 1)) << 19);
                mout[j] = so;
                atomicAdd(&ES->leastCnt[kq - 1], 1);
            } else if (s <= 256) atomicAdd(&ES->hist[s], 1u);
        }
        const uint32_t ntiles = (uint32_t)(((v.out_off - a0) + v.ulen) / DC_TILE) + 2;
#pragma unroll 1
        for (uint32_t t = tid; t < ntiles; t += ENG_NT) tileFirst[t] = v.nm;
        __syncthreads();
#pragma unroll 1
        for (int k = tid; k < 320; k += ENG_NT) litHist[k] = ES->hist[k];
        // tileFirst: match j fills the tiles after its predecessor's up to its own (tiles without a match start included)
#pragma unroll 1
        for (uint32_t j = tid; j < v.nm; j += ENG_NT) {
            const uint32_t ti = (mout[j] - a0) / DC_TILE;
            const uint32_t t0 = j ? (mout[j - 1] - a0) / DC_TILE + 1 : 0u;
#pragma unroll 1
            for (uint32_t t = t0; t <= ti; t++) tileFirst[t] = j;
        }
        // the matches grouped by length symbol (counting sort; the order inside a group does not matter)
        if (tid == 0) {
            uint32_t acc = 0;
#pragma unroll 1
            for (int b = 0; b < 32; b++) { ES->binStart[b] = acc; acc += (uint32_t)ES->leastCnt[b]; ES->leastCnt[b] = (int)ES->binStart[b]; }
            ES->binStart[32] = acc;
            acc = 0;
#pragma unroll 1
            for (int b = 0; b < 32; b++) { ES->itemStart[b] = acc; acc += (ES->binStart[b + 1] - ES->binStart[b] + 31) / 32; }
            ES->itemStart[32] = acc;
        }
        __syncthreads();
#pragma unroll 1
        for (uint32_t j = tid; j < v.nm; j += ENG_NT) perm[atomicAdd(&ES->leastCnt[((minfo[j] >> 14) & 31) - 1], 1)] = j;
        if (tid < 32) {
            uint32_t o = ES->itemStart[tid];
#pragma unroll 1
            for (uint32_t j = ES->binStart[tid]; j < ES->binStart[tid + 1]; j += 32) items[o++] = j | ((uint32_t)tid << 27);
        }
        __syncthreads();
    }

    // symbol-space mask words src -> match-space mask in slot `slot` (bits on symbols that are not matches are dropped)
    __device__ __noinline__ void load_mask(const uint32_t* src, int slot) {
        uint32_t* md = maskp(slot);
#pragma unroll 1
        for (uint32_t k = tid; k < v.nwords; k += ENG_NT) md[k] = 0;
        __syncthreads();
#pragma unroll 1
        for (uint32_t k = tid; k < sym_words(); k += ENG_NT) {
            const uint32_t m = src[k];
            uint32_t f = mflag[k];
            if (!(m & f)) continue;
            uint32_t x = 0;
#pragma unroll 1
            for (int c = 0; f; f &= f - 1, c++) x |= ((m >> (__ffs((int)f) - 1)) & 1u) << c;
            const uint32_t r = mrank[k], sh = r & 31;
            atomicOr(&md[r >> 5], x << sh);
            if (sh && (x >> (32 - sh))) atomicOr(&md[(r >> 5) + 1], x >> (32 - sh));
        }
        __syncthreads();
    }
    // match-space mask in slot `slot` -> symbol-space mask words dst
    __device__ __noinline__ void store_mask(int slot, uint32_t* dst) {
        const uint32_t* ms = maskp(slot);
#pragma unroll 1
        for (uint32_t k = tid; k < sym_words(); k += ENG_NT) {
            uint32_t f = mflag[k], out = 0;
            if (f) {
                const uint32_t r = mrank[k], sh = r & 31, w = r >> 5;
                uint32_t x = ms[w] >> sh;
                if (sh && w + 1 < v.nwords) x |= ms[w + 1] << (32 - sh);
#pragma unroll 1
                for (int c = 0; f; f &= f - 1, c++) out |= ((x >> c) & 1u) << (__ffs((int)f) - 1);
            }
            dst[k] = out;
        }
    }

    // histogram of the symbol list with mask `mid` into ES->hist: the literal histogram plus the matches
    __device__ __noinline__ void pass_hist_full(int mid) {
        P0();
        const uint32_t* m = maskp(mid);
#pragma unroll 1
        for (int k = tid; k < 320; k += ENG_NT) ES->hist[k] = litHist[k];
        __syncthreads();
#pragma unroll 1
        for (uint32_t j = tid; j < v.nm; j += ENG_NT) {
            const uint32_t mi = minfo[j];
            if (!((m[j >> 5] >> (j & 31)) & 1)) {
                atomicAdd(&ES->hist[256 + ((mi >> 14) & 31)], 1u);
                atomicAdd(&ES->hist[288 + ((mi >> 9) & 31)], 1u);
            } else {
                const uint8_t* p = v.out + mout[j];
                const int len = (int)(mi & 0x1FF) + 3;
#pragma unroll 1
                for (int k = 0; k < len; k++) atomicAdd(&ES->hist[p[k]], 1u);
            }
        }
        __syncthreads();
        P1(PR_HIST);
    }

    // payload of the symbol list described by histogram h (global or shared) under table t (recodeToHuffmanInternal,
    // DeflateBlockHuffman.java:759-770); CTA-wide
    __device__ __noinline__ long long hist_payload(const uint32_t* h, const Tab& t) {
        long long acc = 0;
#pragma unroll 1
        for (int k = tid; k < 318; k += ENG_NT) {
            const uint32_t f = h[k];
            if (!f) continue;
            int bits;
            if (k < 257) bits = t.L[k];
            else if (k < 286) bits = t.L[k] + len_ebits_of(k);
            else if (k >= 288) bits = t.D[k - 288] + dist_ebits_of(k - 288);
            else bits = 0;
            acc += (long long)f * bits;
        }
        if (tid == 0) ES->red = 0;
        __syncthreads();
#pragma unroll 1
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if ((tid & 31) == 0 && acc) atomicAdd(&ES->red, (unsigned long long)acc);
        __syncthreads();
        const long long r = (long long)ES->red;
        __syncthreads();
        return r;
    }

    // pools forgotten; tab 0 = the fixed code
    __device__ __noinline__ void reset_pools() {
        __syncthreads();
        sym_reset(ES->sym, tid, ENG_NT);
#pragma unroll 1
        for (int k = tid; k < MAXT; k += ENG_NT) { ES->tabDc[k] = 0xFF; ES->tabLit[k] = 0xFF; }
        if (tid < DCN) ES->dcOwner[tid] = 0xFFFF;
        if (tid < LCN) ES->slotLit[tid] = 0xFF;
        if (tid == 0) { ES->dcNext = 0; ES->nLit = 0; ES->litNext = 0; }
        Tab& f = tabs[TAB_FIXED];
#pragma unroll 1
        for (int k = tid; k < MAX_LL; k += ENG_NT) f.L[k] = (k < 286) ? ((k <= 143) ? 8 : (k <= 255) ? 9 : (k <= 279) ? 7 : 8) : 0;
        if (tid < MAX_D) f.D[tid] = tid < 30 ? 5 : 0;
        if (tid == 0) { f.nL = 286; f.nD = 30; f.type = 1; f.pad[0] = f.pad[1] = f.pad[2] = 0; }
        __syncthreads();
        const unsigned long long h = hash_words((const uint32_t*)&f, (int)(sizeof(Tab) / 4));
        if (tid == 0) { tabHash[0] = h; ES->sym.nTabs = 1; }
        __syncthreads();
    }

    // B := (mask in slot SLOT_B with its histogram in hists[SLOT_B], tables / header / payload of recs[0]); toFixed: the
    // block is first recoded to the fixed code (DeflateBlockHuffman.merge, :1233-1271), payload from the histogram
    __device__ __noinline__ void adopt_B(bool toFixed) {
        reset_pools();
        const uint32_t* ms = maskp(SLOT_B);
        uint32_t* m0 = maskp(0);
#pragma unroll 1
        for (uint32_t k = tid; k < v.nwords; k += ENG_NT) m0[k] = ms[k];
        const uint32_t* hs = histp(SLOT_B);
        uint32_t* h0 = histp(0);
#pragma unroll 1
        for (int k = tid; k < 320; k += ENG_NT) h0[k] = hs[k];
        __syncthreads();
        const unsigned long long h = mask_hash_cta(m0);
        if (tid == 0) { ES->maskHash[0] = h; ES->sym.nMasks = 1; }
        const Cand& src = recs[0];
        SC b;
        b.mid = 0; b.ok = 1; b.hid = -1; b.tabid = TAB_FIXED; b.type = 1;
        long long pay = src.payload;
        if (toFixed) pay = hist_payload(h0, tabs[TAB_FIXED]);
        else if (src.tab.type == 2) {
            uint32_t* st = (uint32_t*)&tabs[MAXT];
            const uint32_t* q = (const uint32_t*)&src.tab;
#pragma unroll 1
            for (int k = tid; k < (int)(sizeof(Tab) / 4); k += ENG_NT) st[k] = q[k];
            uint32_t* hd = (uint32_t*)&hdrs[0];
            const uint32_t* hq = (const uint32_t*)&src.hdr;
#pragma unroll 1
            for (int k = tid; k < (int)(sizeof(Hdr) / 4); k += ENG_NT) hd[k] = hq[k];
            __syncthreads();
            if (tid < 32) {
                const int t = intern_tab_warp(0, tid);
                if (tid == 0) ES->tmpIdx = t;
            }
            __syncthreads();
            b.tabid = (short)ES->tmpIdx; b.type = 2; b.hid = 0;
            if (tid == 0) { ES->sym.hbits[0] = (unsigned short)src.hdr.bits; ES->sym.nHdrs = 1; }
        }
        b.payload = pay;
        if (tid == 0) { ES->en.B = b; ES->en.blockType = b.type; }
        __syncthreads();
    }

    // a new block: symbol view set by the caller, candidate `src` (global), symbol-space mask words `maskSrc`
    __device__ __noinline__ void load_block(const Cand& src, const uint32_t* maskSrc, bool toFixed) {
        P0();
        __syncthreads();
        bigWeights = v.ulen + (uint64_t)v.n + 4 >= (1ull << 22);
#ifdef D4_FORCE_BIG_WEIGHTS   // stress build: every tree takes the slow, exact-weight path
        bigWeights = true;
#endif
        uint32_t* d = (uint32_t*)&recs[0];
        const uint32_t* s = (const uint32_t*)&src;
#pragma unroll 1
        for (int k = tid; k < (int)(sizeof(Cand) / 4); k += ENG_NT) d[k] = s[k];
        build_views();
        load_mask(maskSrc, SLOT_B);
        pass_hist_full(SLOT_B);
        uint32_t* hb = histp(SLOT_B);
#pragma unroll 1
        for (int k = tid; k < 320; k += ENG_NT) hb[k] = ES->hist[k];
        __syncthreads();
        adopt_B(toFixed);
        if (tid == 0) {
            ES->en.trialAll = trialAll;
            ES->tsink.buf = g_trace; ES->tsink.cap = g_trace_cap; ES->tsink.n = &g_trace_n;
            ES->en.trace = g_trace ? &ES->tsink : nullptr;
            ES->en.storedOK = v.ulen <= 65535;
        }
        __syncthreads();
        P1(PR_LOAD);
    }

    // ---- cost arrays ------------------------------------------------------------------------------------------------

    // The cost of a match under table T splits into  lit[i] - refL[length symbol] - refD[distance symbol]:
    //   lit[i]  = sum of the literal code lengths of the match's bytes, DC_BLOCKED when a byte has no code
    //             (DeflateBlockHuffman.java:238-246) - a function of the 256 literal lengths alone.  Most of the tables a
    //             block meets differ in a few length / distance symbols only (measured: 22 of 30 new tables share their
    //             literal lengths with an earlier one), so the arrays are cached per SET OF LITERAL LENGTHS.
    //   refL/D  = code length + extra bits of the two symbols a match is written with: two 32-entry tables per T.
    // Per table only the sign masks (entry < 0, entry == 0) are materialised, by a short streaming pass.

    // refL / refD of table t -> shared memory
    __device__ __forceinline__ void load_ref(int t) {
        const Tab& tb = tabs[t];
        if (tid < 32) ES->refL[tid] = (uint8_t)(tb.L[256 + tid] + (tid > 0 && tid < 30 ? len_ebits_of(256 + tid) : 0));
        else if (tid < 64) ES->refD[tid - 32] = (uint8_t)(tb.D[tid - 32] + (tid - 32 < 30 ? dist_ebits_of(tid - 32) : 0));
    }
    // cost-array entry of match j under the table whose refL / refD are loaded
    __device__ __forceinline__ int dc_val(const short* lit, uint32_t j) const {
        const int x = lit[j];
        if (x == DC_BLOCKED) return DC_BLOCKED;
        const uint32_t mi = minfo[j];
        return x - ES->refL[(mi >> 14) & 31] - ES->refD[(mi >> 9) & 31];
    }

    // the literal-cost array of table t's literal lengths.  ONE coalesced pass over the block's decoded bytes when it is
    // not cached: every warp streams its own run of 512-byte tiles (a 128-bit load per lane, code lengths looked up in
    // shared memory, a warp-wide prefix sum into its slice of shared memory) and every match that starts in a tile takes
    // P[end] - P[start]; the one match that crosses the tile's end is finished from the next tile.  Entry j = match j.
    __device__ __noinline__ const short* ensure_lit(int t) {
        int ls = ES->tabLit[t];
        if (ls == 0xFF) {   // which set of literal lengths is this?
            __syncthreads();
            const uint32_t* q = (const uint32_t*)tabs[t].L;
            unsigned long long hh = 0;
            if (tid < 64) {
                unsigned long long x = (unsigned long long)q[tid] + 0x9E3779B97F4A7C15ull * (unsigned long long)(tid + 1);
                x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
                hh = x;
            }
            const unsigned long long h = cta_sum64(hh);
            if (tid == 0) ES->tmpIdx = -1;
            __syncthreads();
            const int nl = ES->nLit;
#pragma unroll 1
            for (int k = 0; k < nl; k++) {   // few sets: one after the other, confirmed by a full comparison
                if (ES->litHash[k] != h) continue;
                const uint32_t* r = (const uint32_t*)tabs[ES->litRep[k]].L;
                const int diff = __syncthreads_or(tid < 64 && r[tid] != q[tid]);
                if (!diff) { if (tid == 0) ES->tmpIdx = k; break; }
            }
            __syncthreads();
            if (tid == 0) {
                int k = ES->tmpIdx;
                if (k < 0) {
                    if (ES->nLit == MAXLIT) {   // table of sets full: forget all of them (and their arrays)
                        ES->nLit = 0;
                        for (int j = 0; j < MAXT; j++) ES->tabLit[j] = 0xFF;
                        for (int j = 0; j < LCN; j++) ES->slotLit[j] = 0xFF;
                    }
                    k = ES->nLit++;
                    ES->litHash[k] = h; ES->litRep[k] = (unsigned short)t; ES->litSlot[k] = 0xFF;
                }
                ES->tabLit[t] = (unsigned char)k;
            }
            __syncthreads();
            ls = ES->tabLit[t];
        }
        int slot = ES->litSlot[ls];
        if (slot != 0xFF) return dc + (size_t)slot * maxn;
        P0();
        __syncthreads();  // every thread has seen the miss before thread 0 records the new slot
        if (tid == 0) {
            slot = ES->litNext;
            ES->litNext = (slot + 1) % LCN;
            const int owner = ES->slotLit[slot];
            if (owner != 0xFF) ES->litSlot[owner] = 0xFF;
            ES->slotLit[slot] = (unsigned char)ls;
            ES->litSlot[ls] = (unsigned char)slot;
            ES->tmpIdx = slot;
        }
        const Tab& tb = tabs[t];
#pragma unroll 1
        for (int k = tid; k < 256; k += ENG_NT) { const uint32_t c = tb.L[k]; ES->ctab[k] = c ? c : 0x10000u; }
        __syncthreads();
        slot = ES->tmpIdx;
        short* d = dc + (size_t)slot * maxn;
        const uint32_t a0 = (uint32_t)(v.out_off & ~15ull);
        const uint32_t head = (uint32_t)(v.out_off - a0);
        const uint32_t endRel = head + (uint32_t)v.ulen;
        const uint8_t* base = v.out + a0;
        const int lane = tid & 31, wid = tid >> 5;
        uint32_t* P = ES->u.P[wid];
        const uint32_t ntiles = endRel / DC_TILE + 1;
        const uint32_t per = (ntiles + ENG_NW - 1) / ENG_NW;
        const uint32_t T0 = (uint32_t)wid * per, T1 = min(ntiles, T0 + per);
        // Software pipeline, one tile deep: while tile T is processed, the bytes of T+1, the match range of T+2 and the
        // first DC_PRE * 32 match records of T+1 are already in flight; the match that crosses from T into T+1 travels in
        // lane 0's registers.  P[k] holds the prefix of byte k relative to its lane's first byte, LB[l] the prefix of lane
        // l's first byte: the prefix at byte k is LB[k / 16] + P[k] (P[DC_TILE] = 0, LB[32] = tile total).
        constexpr int DC_PRE = 4;
        uint32_t* LB = P + DC_TILE + 4;
        int carryIdx = -1;
        uint32_t carryPart = 0, carryEnd = 0;
        uint4 q = make_uint4(0, 0, 0, 0);
        uint32_t i0 = 0, i1 = 0, i2 = 0;       // matches of the current tile: [i0, i1); of the next one: [i1, i2)
        uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0;
        if (T0 < T1) {
            const uint32_t idx = T0 * DC_TILE + 16u * (uint32_t)lane;
            if (idx < endRel) q = *(const uint4*)(base + idx);
            i0 = tileFirst[T0]; i1 = tileFirst[T0 + 1];
            i2 = (T0 + 1 < T1) ? tileFirst[T0 + 2] : i1;
            const uint32_t i = i0 + (uint32_t)lane;
            m0 = i < i1 ? minfo[i] : 0u; m1 = i + 32 < i1 ? minfo[i + 32] : 0u;
            m2 = i + 64 < i1 ? minfo[i + 64] : 0u; m3 = i + 96 < i1 ? minfo[i + 96] : 0u;
        }
        if (lane == 0) P[DC_TILE] = 0;
#define D4_PFX(k) (LB[(k) >> 4] + P[(k)])
        // one match record (0: none): a match inside the tile gets its literal cost, the one that crosses the tile's end is
        // remembered
#define D4_DC_ONE(i_, m_)                                                                                        \
        do {                                                                                                     \
            const uint32_t mm = (m_);                                                                            \
            if ((mm >> 14) & 31) {                                                                               \
                const uint32_t s0 = (mm >> 19) & (DC_TILE - 1), e = s0 + (mm & 0x1FF) + 3;                       \
                if (e <= DC_TILE) {                                                                              \
                    const uint32_t y = D4_PFX(e) - D4_PFX(s0);                                                   \
                    d[(i_)] = (y >> 16) ? DC_BLOCKED : (short)(y & 0xffffu);                                     \
                } else { nIdx = (int)(i_); nPart = LB[32] - D4_PFX(s0); nEnd = e - DC_TILE; }                    \
            }                                                                                                    \
        } while (0)
        // one tile past the warp's run finishes its last crossing match
#pragma unroll 1
        for (uint32_t T = T0; T <= T1 && T <= ntiles; T++) {
            const bool extra = T >= T1;
            if (extra && __shfl_sync(0xffffffffu, carryIdx, 0) < 0) break;
            const uint32_t idx = T * DC_TILE + 16u * (uint32_t)lane;
            const uint4 cur = q;
            const uint32_t ci0 = i0, ci1 = i1;
            const uint32_t c0 = m0, c1 = m1, c2 = m2, c3 = m3;
            if (T + 1 <= T1 && T + 1 <= ntiles) {   // next tile: its bytes, its first match records, the range after it
                const uint32_t nidx = idx + DC_TILE;
                q = (nidx < endRel) ? *(const uint4*)(base + nidx) : make_uint4(0, 0, 0, 0);
                i0 = ci1; i1 = i2;
                i2 = (T + 2 < T1) ? tileFirst[T + 3] : i1;
                if (T + 1 < T1) {
                    const uint32_t i = i0 + (uint32_t)lane;
                    m0 = i < i1 ? minfo[i] : 0u; m1 = i + 32 < i1 ? minfo[i + 32] : 0u;
                    m2 = i + 64 < i1 ? minfo[i + 64] : 0u; m3 = i + 96 < i1 ? minfo[i + 96] : 0u;
                }
            }
            // per-byte costs -> lane-relative exclusive prefixes straight into shared memory, 4 at a time
            uint32_t run = 0;
            const bool inside = T * DC_TILE >= head && (T + 1) * DC_TILE <= endRel;   // no per-byte bounds inside the block
#pragma unroll
            for (int g = 0; g < 4; g++) {
                const uint32_t w = g == 0 ? cur.x : g == 1 ? cur.y : g == 2 ? cur.z : cur.w;
                uint4 o;
                uint32_t x0 = ES->ctab[w & 0xffu], x1 = ES->ctab[(w >> 8) & 0xffu], x2 = ES->ctab[(w >> 16) & 0xffu], x3 = ES->ctab[w >> 24];
                if (!inside) {
                    const uint32_t j = idx + 4 * g;
                    if (!(j >= head && j < endRel)) x0 = 0;
                    if (!(j + 1 >= head && j + 1 < endRel)) x1 = 0;
                    if (!(j + 2 >= head && j + 2 < endRel)) x2 = 0;
                    if (!(j + 3 >= head && j + 3 < endRel)) x3 = 0;
                }
                o.x = run; run += x0;
                o.y = run; run += x1;
                o.z = run; run += x2;
                o.w = run; run += x3;
                *(uint4*)(P + 16 * lane + 4 * g) = o;
            }
            uint32_t incl = run;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, incl, dd);
                if (lane >= dd) incl += y;
            }
            LB[lane] = incl - run;
            if (lane == 31) LB[32] = incl;
            __syncwarp();
            if (lane == 0 && carryIdx >= 0) {
                const uint32_t y = carryPart + D4_PFX(carryEnd);
                d[carryIdx] = (y >> 16) ? DC_BLOCKED : (short)(y & 0xffffu);
                carryIdx = -1;
            }
            if (!extra) {
                int nIdx = -1;
                uint32_t nPart = 0, nEnd = 0;
                const uint32_t ib = ci0 + (uint32_t)lane;
                D4_DC_ONE(ib, c0);
                D4_DC_ONE(ib + 32, c1);
                D4_DC_ONE(ib + 64, c2);
                D4_DC_ONE(ib + 96, c3);
#pragma unroll 1
                for (uint32_t i = ib + 32u * DC_PRE; i < ci1; i += 32) { const uint32_t mx = minfo[i]; D4_DC_ONE(i, mx); }   // many short matches
                // hand the crossing match (if any) to lane 0
                const unsigned who = __ballot_sync(0xffffffffu, nIdx >= 0);
                if (who) {
                    const int src = __ffs((int)who) - 1;
                    carryIdx = __shfl_sync(0xffffffffu, nIdx, src);
                    carryPart = __shfl_sync(0xffffffffu, nPart, src);
                    carryEnd = __shfl_sync(0xffffffffu, nEnd, src);
                }
            }
            __syncwarp();
        }
#undef D4_DC_ONE
#undef D4_PFX
        __syncthreads();
        P1(PR_DC);
        return d;
    }

    // the sign masks of table t's cost array: bit j of negW / zerW = entry j is negative / zero.  One streaming pass over
    // the literal costs and the match records, eight matches (one mask byte) per thread and step.  Leaves refL / refD of
    // t in shared memory.
    __device__ __noinline__ const uint32_t* ensure_masks(int t, const short* lit) {
        load_ref(t);
        int slot = ES->tabDc[t];
        __syncthreads();
        if (slot != 0xFF) return dcBits + (size_t)slot * 2 * maxwords;
        P0();
        if (tid == 0) {
            slot = ES->dcNext;
            ES->dcNext = (slot + 1) % DCN;
            const int owner = ES->dcOwner[slot];
            if (owner != 0xFFFF) ES->tabDc[owner] = 0xFF;
            ES->dcOwner[slot] = (unsigned short)t;
            ES->tabDc[t] = (unsigned char)slot;
            ES->tmpIdx = slot;
        }
        __syncthreads();
        slot = ES->tmpIdx;
        uint32_t* negW = dcBits + (size_t)slot * 2 * maxwords;
        uint8_t* negB = (uint8_t*)negW;
        uint8_t* zerB = (uint8_t*)(negW + maxwords);
        const uint32_t end = v.nwords * 32, nm = v.nm;
        uint32_t j0 = (uint32_t)tid * 8;
        uint4 lq = make_uint4(0, 0, 0, 0), mq0 = lq, mq1 = lq;
        if (j0 < nm) { lq = *(const uint4*)(lit + j0); mq0 = *(const uint4*)(minfo + j0); mq1 = *(const uint4*)(minfo + j0 + 4); }
#pragma unroll 1
        while (j0 < end) {
            const uint4 cl = lq, c0 = mq0, c1 = mq1;
            const uint32_t nx = j0 + ENG_NT * 8;
            if (nx < nm) { lq = *(const uint4*)(lit + nx); mq0 = *(const uint4*)(minfo + nx); mq1 = *(const uint4*)(minfo + nx + 4); }
            uint32_t nb = 0, zb = 0;
            if (j0 < nm) {
                const uint32_t lw[4] = {cl.x, cl.y, cl.z, cl.w}, mw[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int x = (int)(short)((u & 1) ? (lw[u >> 1] >> 16) : (lw[u >> 1] & 0xffffu));
                    if (j0 + u < nm && x != DC_BLOCKED) {
                        const int val = x - ES->refL[(mw[u] >> 14) & 31] - ES->refD[(mw[u] >> 9) & 31];
                        nb |= (val < 0 ? 1u : 0u) << u;
                        zb |= (val == 0 ? 1u : 0u) << u;
                    }
                }
            }
            negB[j0 >> 3] = (uint8_t)nb;
            zerB[j0 >> 3] = (uint8_t)zb;
            j0 = nx;
        }
        __syncthreads();
        P1(PR_MASKS);
        return negW;
    }

    // match j leaves the symbol list and its bytes enter it as literals: histogram delta in ES->hist
    __device__ __noinline__ void hist_delta_replace(uint32_t j) {
        const uint32_t mi = minfo[j];
        atomicSub(&ES->hist[256 + ((mi >> 14) & 31)], 1u);
        atomicSub(&ES->hist[288 + ((mi >> 9) & 31)], 1u);
        const uint8_t* p = v.out + mout[j];
        const int len = (int)(mi & 0x1FF) + 3;
#pragma unroll 1
        for (int k = 0; k < len; k++) atomicAdd(&ES->hist[p[k]], 1u);
    }
    // The same for every match a pass has just replaced, with the whole CTA: the pass queues the matches, then a thread
    // per short match (its bytes loaded eight at a time) and a warp per long one apply the delta.
    // all 32 lanes call this together with the matches (bits of `nbits`, ranks i0 ..) each of them replaced in this step:
    // one shared-memory atomic per warp and step instead of one per match
    __device__ __noinline__ void hq_push_warp(uint32_t nbits, uint32_t i0, int lane) {
        const uint32_t cnt = (uint32_t)__popc(nbits);
        uint32_t incl = cnt;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, incl, dd); if (lane >= dd) incl += y; }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        if (!total) return;
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&ES->u.hq.nS, total);
        base = __shfl_sync(0xffffffffu, base, 0) + incl - cnt;
#pragma unroll 1
        for (uint32_t b = nbits; b; b &= b - 1, base++) {
            const uint32_t i = i0 + (uint32_t)__ffs((int)b) - 1;
            if (base < HQS) ES->u.hq.qs[base] = i;
            else {   // queue full: this one is applied on the spot
                hist_delta_replace(i);
                if (ES->hqLit) atomicAdd(&ES->red, (unsigned long long)(long long)(-dc_val(ES->hqLit, i)));
            }
        }
    }
    // `lit` (replace passes): the cost-array entries of the queued matches are summed into ES->red on the way (what the
    // replacements save); nullptr: not wanted
    __device__ __noinline__ void hq_apply(const short* lit) {
        __syncthreads();
        const uint32_t nS = min(ES->u.hq.nS, (uint32_t)HQS);
        long long sv = 0;
#pragma unroll 1
        for (uint32_t j = tid; j < nS; j += ENG_NT) {
            const uint32_t i = ES->u.hq.qs[j];
            const uint32_t mi = minfo[i];
            const uint32_t so = mout[i];
            if (lit) sv -= dc_val(lit, i);
            const int len = (int)(mi & 0x1FF) + 3;
            atomicSub(&ES->hist[256 + ((mi >> 14) & 31)], 1u);
            atomicSub(&ES->hist[288 + ((mi >> 9) & 31)], 1u);
            if (len > 24) {
                const uint32_t k = atomicAdd(&ES->u.hq.nL, 1u);
                if (k < HQL) { ES->u.hq.ql[k] = i; continue; }
            }
            const uint8_t* p = v.out + so;
#pragma unroll 1
            for (int k = 0; k < len; k += 8) {
                uint32_t b[8];
#pragma unroll
                for (int q = 0; q < 8; q++) b[q] = (k + q < len) ? (uint32_t)p[k + q] : 256u;
#pragma unroll
                for (int q = 0; q < 8; q++) if (b[q] < 256u) atomicAdd(&ES->hist[b[q]], 1u);
            }
        }
        if (lit) {
#pragma unroll
            for (int dd = 16; dd > 0; dd >>= 1) sv += __shfl_xor_sync(0xffffffffu, sv, dd);
            if ((tid & 31) == 0 && sv) atomicAdd(&ES->red, (unsigned long long)sv);
        }
        __syncthreads();
        const uint32_t nL = min(ES->u.hq.nL, (uint32_t)HQL);
        const int lane = tid & 31;
#pragma unroll 1
        for (uint32_t j = (uint32_t)(tid >> 5); j < nL; j += ENG_NW) {
            const uint32_t i = ES->u.hq.ql[j];
            const int len = (int)(minfo[i] & 0x1FF) + 3;
            const uint8_t* p = v.out + mout[i];
#pragma unroll 1
            for (int k = lane; k < len; k += 32) atomicAdd(&ES->hist[p[k]], 1u);
        }
        __syncthreads();
    }
    // hists[dst] = hists[src] + ES->hist (the delta of the matches that were just replaced)
    __device__ __forceinline__ void hist_store_delta(int dst, int src) {
        const uint32_t* hs = histp(src);
        uint32_t* hd = histp(dst);
#pragma unroll 1
        for (int k = tid; k < 320; k += ENG_NT) hd[k] = hs[k] + ES->hist[k];
    }

    // replaceBackrefsWithLiteralsIfSmaller(prune) for memo slot `slot` = (mid, tabid): the candidates are the matches
    // whose cost-array entry is negative (prune: not positive) and that the mask does not cover yet - one AND of the
    // cost array's sign words with the mask words, a word (32 matches) per thread and step; the entries themselves are
    // only read for the (few) matches that are replaced.
    __device__ __noinline__ void pass_replace(int slot, int mid, int tabid, bool prune) {
        if (ES->sym.nMasks >= MAXM) { if (tid == 0) ES->sym.overflow = 1; __syncthreads(); return; }
        const short* d = ensure_lit(tabid);
        const uint32_t* negW = ensure_masks(tabid, d);   // (also loads the table's refL / refD)
        const uint32_t* zerW = negW + maxwords;
        P0();
#pragma unroll 1
        for (int k = tid; k < 320; k += ENG_NT) ES->hist[k] = 0;
        if (tid == 0) { ES->red = 0; ES->redAny = 0; ES->u.hq.nS = 0; ES->u.hq.nL = 0; ES->hqLit = d; }
        __syncthreads();
        const int fresh = ES->sym.nMasks;
        const uint32_t* mo = maskp(mid);
        uint32_t* mn = maskp(fresh);
        unsigned long long hsh = 0;
        const int lane = tid & 31;
        bool any = false;
#pragma unroll 1
        for (uint32_t kb = (uint32_t)(tid & ~31); kb < v.nwords; kb += ENG_NT) {   // per warp: every lane stays for the queue push
            const uint32_t k = kb + (uint32_t)lane;
            uint32_t cand = 0;
            if (k < v.nwords) {
                const uint32_t m = mo[k];
                cand = (negW[k] | (prune ? zerW[k] : 0u)) & ~m;
                mn[k] = m | cand;
                if (cand) {
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const uint32_t b0 = (m >> (8 * q)) & 0xffu, b1 = ((m | cand) >> (8 * q)) & 0xffu;
                        if (b0 != b1) hsh += mask_byte_hash(b1, 4 * k + q) - mask_byte_hash(b0, 4 * k + q);
                    }
                }
            }
            if (__any_sync(0xffffffffu, cand != 0)) { hq_push_warp(cand, 32 * k, lane); any |= cand != 0; }
        }
        if (any) ES->redAny = 1;
        const unsigned long long h = ES->maskHash[mid] + cta_sum64(hsh);   // (also the barrier after the loop)
        __syncthreads();
        P1(PR_PASS_MAIN);
        int newmid = mid;
        if (ES->redAny) {
            { P0(); hq_apply(d); P1(PR_PASS_HQ); }
            newmid = intern_mask(h);
            if (newmid == fresh) hist_store_delta(newmid, mid);
        }
        if (tid == 0) {
            PSlot& p = ES->sym.pm[slot];
            p.mid = (unsigned short)newmid; p.delta = (long long)ES->red; p.state = ST_DONE;
            // recodeHuffmanLessMatches (DeflateBlockHuffman.java:655-658) is the only user of the pruning pass and recodes
            // its result right away: ask for that now, so it runs in this very step
            if (prune && ES->sym.rc[newmid].state == ST_EMPTY) ES->sym.rc[newmid].state = ST_PENDING;
        }
        __syncthreads();
    }

    // removeDistLitLeastExpensive (DeflateBlockHuffman.java:373-458) on (mid, tabid) for memo slot slot0 (mode 0: least
    // cost sum) and / or slot1 (mode 1: least count); a slot < 0 is not wanted.  The statistics are the same for both
    // modes, so a state that asks for both pays for them once.  They are taken over the block's matches grouped by
    // length symbol (perm / binStart): every thread walks a contiguous stretch of that list and adds its partial sums
    // to the shared bins when the length symbol changes - a handful of atomics per thread, no warp-wide voting.
    __device__ __noinline__ void pass_least(int slot0, int slot1, int mid, int tabid) {
        if (ES->sym.nMasks + 2 > MAXM) { if (tid == 0) ES->sym.overflow = 1; __syncthreads(); return; }
        const short* d = ensure_lit(tabid);
        load_ref(tabid);
        P0();
        if (tid < 32) { ES->leastSum[tid] = 0; ES->leastCnt[tid] = 0; }
        if (tid == 0) { ES->leastBlocked = 0; ES->leastSeen = 0; }
        __syncthreads();
        const int lane = tid & 31;
        const uint8_t* mbytes = (const uint8_t*)maskp(mid);
        {
            const uint32_t nItems = ES->itemStart[32];
#pragma unroll 1
            for (uint32_t it = tid; it < nItems; it += ENG_NT) {   // <= 32 matches of one length symbol per item
                const uint32_t w = items[it];
                const int bin = (int)(w >> 27);
                uint32_t j = w & 0x7FFFFFFu;
                const uint32_t jend = min(ES->binStart[bin + 1], j + 32);
                int sum = 0, cnt = 0;
                bool blocked = false, seen = false;
#pragma unroll 1
                for (; j < jend; j += 8) {   // eight matches at a time: indices, then costs and mask bytes, in flight together
                    uint32_t idx[8];
                    int xv[8];
                    uint32_t mk[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) idx[u] = j + u < jend ? perm[j + u] : 0u;
#pragma unroll
                    for (int u = 0; u < 8; u++) { xv[u] = d[idx[u]]; mk[u] = mbytes[idx[u] >> 3] | (minfo[idx[u]] & (31u << 9)); }
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const bool live = j + u < jend && !((mk[u] >> (idx[u] & 7)) & 1);   // still a match
                        seen |= live;
                        const bool blk = live && xv[u] == DC_BLOCKED;
                        blocked |= blk;
                        if (live && !blk) { sum += xv[u] - ES->refL[bin + 1] - ES->refD[mk[u] >> 9]; cnt++; }
                    }
                }
                if (seen) atomicOr(&ES->leastSeen, 1u << bin);
                if (blocked) atomicOr(&ES->leastBlocked, 1u << bin);
                if (cnt) { atomicAdd(&ES->leastSum[bin], sum); atomicAdd(&ES->leastCnt[bin], cnt); }
            }
        }
        __syncthreads();
        if (tid == 0) {
#pragma unroll 1
            for (int mode = 0; mode < 2; mode++) {
                int rem = -1, remSize = 0, remFreq = 0;
#pragma unroll 1
                for (int i = 0; i < 32; i++) {
                    if (!((ES->leastBlocked >> i) & 1) && ((ES->leastSeen >> i) & 1)) {
                        bool doRem = mode == 1 ? ES->leastCnt[i] < remFreq : ES->leastSum[i] < remSize;
                        if (rem == -1 || doRem) { rem = i; remSize = ES->leastSum[i]; remFreq = ES->leastCnt[i]; }
                    }
                }
                ES->leastRem[mode] = rem; ES->leastSize[mode] = remSize;
            }
        }
        __syncthreads();
        P1(PR_PASS_LEAST);
        int doneMid = -1, doneRem = -2;
#pragma unroll 1
        for (int mode = 0; mode < 2; mode++) {
            const int slot = mode ? slot1 : slot0;
            if (slot < 0) continue;
            const int rem = ES->leastRem[mode];
            int newmid = mid;
            if (rem >= 0 && rem == doneRem) newmid = doneMid;   // both modes remove the same length symbol
            else if (rem >= 0) {
                P0();
#pragma unroll 1
                for (int k = tid; k < 320; k += ENG_NT) ES->hist[k] = 0;
                if (tid == 0) { ES->u.hq.nS = 0; ES->u.hq.nL = 0; ES->hqLit = nullptr; }
                const int fresh = ES->sym.nMasks;
                const uint32_t* mo = maskp(mid);
                uint32_t* mn = maskp(fresh);
#pragma unroll 1
                for (uint32_t k = tid; k < v.nwords; k += ENG_NT) mn[k] = mo[k];
                __syncthreads();
                // every match of the length symbol that is still a match: mask bit + histogram queue
                const uint32_t j0 = ES->binStart[rem], j1 = ES->binStart[rem + 1];
#pragma unroll 1
                for (uint32_t jb = j0 + (uint32_t)(tid & ~31); jb < j1; jb += ENG_NT) {   // warp-uniform trip count
                    const uint32_t j = jb + (uint32_t)lane;
                    uint32_t i = 0;
                    bool fresh1 = false;
                    if (j < j1) {
                        i = perm[j];
                        fresh1 = !((mbytes[i >> 3] >> (i & 7)) & 1);
                        if (fresh1) atomicOr(&mn[i >> 5], 1u << (i & 31));
                    }
                    // queue the newly replaced matches of this warp with one shared atomic
                    const unsigned bal = __ballot_sync(0xffffffffu, fresh1);
                    if (bal) {
                        uint32_t base = 0;
                        if (lane == 0) base = atomicAdd(&ES->u.hq.nS, (uint32_t)__popc(bal));
                        base = __shfl_sync(0xffffffffu, base, 0) + (uint32_t)__popc(bal & ((1u << lane) - 1u));
                        if (fresh1) { if (base < HQS) ES->u.hq.qs[base] = i; else hist_delta_replace(i); }
                    }
                }
                __syncthreads();
                // the mask hash moves by the bytes that changed
                unsigned long long hsh = 0;
#pragma unroll 1
                for (uint32_t k = tid; k < v.nwords; k += ENG_NT) {
                    const uint32_t a0 = mo[k], a1 = mn[k];
                    if (a0 == a1) continue;
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const uint32_t b0 = (a0 >> (8 * q)) & 0xffu, b1 = (a1 >> (8 * q)) & 0xffu;
                        if (b0 != b1) hsh += mask_byte_hash(b1, 4 * k + q) - mask_byte_hash(b0, 4 * k + q);
                    }
                }
                const unsigned long long h = ES->maskHash[mid] + cta_sum64(hsh);
                hq_apply(nullptr);
                newmid = intern_mask(h);
                if (newmid == fresh) hist_store_delta(newmid, mid);
                doneMid = newmid; doneRem = rem;
                P1(PR_LEAST_APPLY);
            }
            if (tid == 0) {
                PSlot& p = ES->sym.pm[slot];
                p.mid = (unsigned short)newmid; p.delta = -(long long)ES->leastSize[mode]; p.state = ST_DONE;
            }
            __syncthreads();
        }
    }

    __device__ __noinline__ void exec_passes() {
        const int nq = ES->sym.nqPass;
        if (!nq) return;
        P0();
#pragma unroll 1
        for (int q = 0; q < nq; q++) {
            const int slot = ES->sym.qPass[q];
            const unsigned key = ES->sym.pm[slot].key;
            const int mid = pm_key_mid(key), tabid = pm_key_tab(key), op = pm_key_op(key);
            if (ES->sym.pm[slot].state == ST_DONE) continue;   // done together with its sibling (least passes)
            if (op == OP_FIXED) {   // recodeToFixedHuffman: the fixed-code payload is a function of the symbol list alone
                const long long pay = hist_payload(histp(mid), tabs[TAB_FIXED]);
                if (tid == 0) { PSlot& p = ES->sym.pm[slot]; p.delta = pay; p.mid = (unsigned short)mid; p.state = ST_DONE; }
                __syncthreads();
            } else if (op <= OP_REPLACE_PRUNE) pass_replace(slot, mid, tabid, op == OP_REPLACE_PRUNE);
            else {
                // the other mode on the same state, when it is waiting too
                const unsigned sib = pm_key(mid, tabid, op == OP_LEAST0 ? OP_LEAST1 : OP_LEAST0);
                int other = -1;
#pragma unroll 1
                for (int r = q + 1; r < nq; r++)
                    if (ES->sym.pm[ES->sym.qPass[r]].key == sib && ES->sym.pm[ES->sym.qPass[r]].state != ST_DONE) { other = ES->sym.qPass[r]; break; }
                pass_least(op == OP_LEAST0 ? slot : other, op == OP_LEAST0 ? other : slot, mid, tabid);
            }
        }
        // a pass that could not run (mask pool full) leaves its slot pending: the round restarts after a reset
        PCOUNT(PR_PASS, nq - 1);
        P1(PR_PASS);
    }

    // ---- recodeHuffman, one warp per request ------------------------------------------------------------------------
    // runs of equal code lengths of a Tab, cut by one warp: ballot + popcount compaction (`start`: MAX_PAIRS scratch)
    static __device__ __forceinline__ void runlist_warp(const Tab& t, RunList& rl, uint16_t* start, int lane) {
        const int nL = t.nL, n = t.nL + t.nD;
        int cnt = 0;
#pragma unroll 1
        for (int i0 = 0; i0 < n; i0 += 32) {
            const int i = i0 + lane;
            const int vv = i < n ? (i < nL ? t.L[i] : t.D[i - nL]) : -1;
            const int pv = (i > 0 && i < n) ? (i - 1 < nL ? t.L[i - 1] : t.D[i - 1 - nL]) : -2;
            const bool st = i < n && vv != pv;
            const unsigned bal = __ballot_sync(0xffffffffu, st);
            if (st) {
                const int k = cnt + __popc(bal & ((1u << lane) - 1u));
                rl.val[k] = (uint8_t)vv;
                start[k] = (uint16_t)i;
            }
            cnt += __popc(bal);
        }
        __syncwarp();
#pragma unroll 1
        for (int k = lane; k < cnt; k += 32) rl.len[k] = (uint16_t)((k + 1 < cnt ? start[k + 1] : n) - start[k]);
        if (lane == 0) rl.n = (uint16_t)cnt;
        __syncwarp();
    }

    // header code of the pair frequencies f[0..19) (Huffman.ofRLEPacked), trimmed on from `ncl`, and the header size:
    // sum of pair bits = sum_s freq[s] * CL[s] + 2 f16 + 3 f17 + 7 f18.  One thread.
    __device__ __noinline__ void hdr_code_from_freq(const uint32_t* f, uint8_t* CL, int ncl, int* nclOut, int* bitsOut, unsigned char* wsb) {
        // fast path in 100 bytes, the full algorithm (compact workspace) behind it
        TreeWsTiny ws{reinterpret_cast<uint16_t*>(wsb), wsb + 48, reinterpret_cast<TreeWsCLc*>(wsb + 104)};
        if (huff_tree_ws(f, 19, 7, CL, ws)) ES->err = ERR_TREE;
        ncl = trim_ncl(CL, ncl);
        int bits = 5 + 5 + 4 + 3 * ncl + 2 * (int)f[16] + 3 * (int)f[17] + 7 * (int)f[18];
#pragma unroll 1
        for (int k = 0; k < 19; k++) bits += (int)f[k] * CL[k];
        *nclOut = ncl;
        *bitsOut = bits;
    }

    // rewriteHeader with the default strategy (DeflateBlockHuffman.java:480-577) for table `t` into header `h` (both
    // global), by one warp: runs -> pairs per run -> exclusive scan -> every run writes its pairs
    __device__ __noinline__ void hdr_default_warp(const Tab& t, Hdr& h, unsigned char* wsb, int lane) {
        RunList& rl = *reinterpret_cast<RunList*>(wsb);
        uint16_t* start = reinterpret_cast<uint16_t*>(wsb + 964);         // MAX_PAIRS
        uint16_t* off = reinterpret_cast<uint16_t*>(wsb + 1608);          // MAX_PAIRS + 2
        uint32_t* f19 = reinterpret_cast<uint32_t*>(wsb + 2256);          // 19 (+ CL staging)
        uint8_t* cl = wsb + 2336;                                          // 19
        unsigned char* tw = wsb + 2368;
        static_assert(sizeof(RunList) <= 964 && 964 + 2 * MAX_PAIRS <= 1608 && 2368 + 104 + sizeof(TreeWsCLc) <= WS_BYTES, "warp workspace layout");
        if (lane < 19) f19[lane] = 0;
        runlist_warp(t, rl, start, lane);
        const int R = rl.n;
#pragma unroll 1
        for (int r = lane; r < R; r += 32) {
            int cnt = 0;
            emit_run(rl.val[r], rl.len[r], FLAGS_DEFAULT, [&](int, int, int, int k) { cnt += k; });
            off[r] = (uint16_t)cnt;
        }
        __syncwarp();
        int carry = 0;
#pragma unroll 1
        for (int i0 = 0; i0 < R; i0 += 32) {
            const int i = i0 + lane;
            const int x = i < R ? off[i] : 0;
            int incl = x;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, dd); if (lane >= dd) incl += y; }
            if (i < R) off[i] = (uint16_t)(carry + incl - x);
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        __syncwarp();
#pragma unroll 1
        for (int r = lane; r < R; r += 32) {
            int o = off[r];
            emit_run(rl.val[r], rl.len[r], FLAGS_DEFAULT, [&](int sym, int run, int val, int k) {
                const uint16_t p = pair_pack(sym, run, val);
#pragma unroll 1
                for (int q = 0; q < k; q++) h.pairs[o++] = p;
                atomicAdd(&f19[sym], (uint32_t)k);
            });
        }
        __syncwarp();
        if (lane == 0) {
            int ncl, bits;
            hdr_code_from_freq(f19, cl, 19, &ncl, &bits, tw);
            h.np = (uint16_t)carry; h.ncl = (uint8_t)ncl; h.bits = bits;
#pragma unroll 1
            for (int k = 0; k < 19; k++) h.CL[k] = cl[k];
        }
        __syncwarp();
    }

    __device__ __noinline__ void recode_one(int mid, int w, int lane, int hid) {
        unsigned char* wsb = ES->u.ws[w];
        uint32_t* heap = reinterpret_cast<uint32_t*>(wsb);                 // 294 words (also the distance tree workspace)
        uint32_t* freq = reinterpret_cast<uint32_t*>(wsb + 1184);          // 320 words; the litlen tree's parent[] later
        uint16_t* value = reinterpret_cast<uint16_t*>(wsb + 2464);         // 292
        static_assert(sizeof(TreeWs<32, 68>) <= 1184 && 2464 + 292 * 2 <= WS_BYTES, "warp workspace layout");
        const uint32_t* hs = histp(mid);
#pragma unroll 1
        for (int k = lane; k < 320; k += 32) freq[k] = hs[k];
        Tab& T = tabs[MAXT + w];
#pragma unroll 1
        for (int k = lane; k < MAX_LL; k += 32) T.L[k] = 0;
        T.D[lane] = 0;
        __syncwarp();
        P0();
        uint32_t nr = 0;
        int nl = 286;
        if (lane == 0) {
            // trailing zero-frequency trimming + the distance special cases (DeflateBlockHuffman.java:683-740)
            const uint32_t* df = freq + 288;
            int nd = 30;
            while (nd > 0 && df[nd - 1] == 0) nd--;
            int nz = 0;
#pragma unroll 1
            for (int k = 0; k < nd; k++) nz += df[k] != 0;
            if (nd == 0) { T.nD = 1; }                                          // handleZero: one entry, length 0
            else if (nz <= 1) { T.nD = (uint16_t)nd; T.D[nd - 1] = 1; }         // handleOne
            else {
                T.nD = (uint16_t)nd;
                int deepD = 16;
                if (!bigWeights) {   // same fast path as the litlen tree (the distance counts die with it: parent[] overlays them)
                    uint16_t* valD = reinterpret_cast<uint16_t*>(wsb + 512);
                    const uint32_t nrD = huff_tree_fast_build(freq + 288, nd, heap, valD);
                    deepD = huff_tree_fast_depths(reinterpret_cast<const uint16_t*>(freq + 288), valD, nd, nrD, T.D, 0, 1);
                }
                if (deepD > 15) {
#pragma unroll 1
                    for (int k = 0; k < MAX_D; k++) T.D[k] = 0;
                    if (huff_tree<32, 68>(hs + 288, nd, 15, T.D, *reinterpret_cast<TreeWs<32, 68>*>(wsb))) ES->err = ERR_TREE;
                }
            }
            while (nl > 0 && freq[nl - 1] == 0) nl--;
            T.nL = (uint16_t)nl;
            T.type = 2; T.pad[0] = T.pad[1] = T.pad[2] = 0;
            if (!bigWeights) nr = huff_tree_fast_build(freq, nl, heap, value);
        }
        nr = __shfl_sync(0xffffffffu, nr, 0);
        nl = __shfl_sync(0xffffffffu, nl, 0);
        int deep = 16;
        if (!bigWeights) {   // code lengths: every lane walks some leaves up to the root
            deep = huff_tree_fast_depths(reinterpret_cast<const uint16_t*>(freq), value, nl, nr, T.L, lane, 32);
#pragma unroll 1
            for (int dd = 16; dd > 0; dd >>= 1) deep = max(deep, __shfl_xor_sync(0xffffffffu, deep, dd));
        }
        if (deep > 15) {   // deeper than 15 (or weights too large for the fast keys): the full algorithm with its limiter
            __syncwarp();
#pragma unroll 1
            for (int k = lane; k < MAX_LL; k += 32) T.L[k] = 0;
            __syncwarp();
            if (lane == 0) {
                PCOUNT(PR_SLOWTREE, 1);
                if (huff_tree<290, 584>(hs, nl, 15, T.L, slowWs[w])) ES->err = ERR_TREE;
            }
        }
        __syncwarp();
        P1(PR_TREES);
        // payload = histogram . (code length + extra bits) (recodeToHuffmanInternal, :759-770)
        long long acc = 0;
#pragma unroll 1
        for (int k = lane; k < 318; k += 32) {
            const uint32_t f = hs[k];
            if (!f) continue;
            int bits;
            if (k < 257) bits = T.L[k];
            else if (k < 286) bits = T.L[k] + len_ebits_of(k);
            else if (k >= 288) bits = T.D[k - 288] + dist_ebits_of(k - 288);
            else bits = 0;
            acc += (long long)f * bits;
        }
#pragma unroll 1
        for (int dd = 16; dd > 0; dd >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, dd);
        if (lane == 0) ES->recPay[w] = acc;
        const long long p1_ = clock64();
        hdr_default_warp(T, hdrs[hid], wsb, lane);
        { const long long p0_ = p1_; (void)p0_; P1(PR_HDR_DEFAULT); }
        if (lane == 0) ES->sym.hbits[hid] = (unsigned short)hdrs[hid].bits;
        __syncwarp();
    }

    __device__ __noinline__ void exec_recodes() {
        const int nq = ES->sym.nqRec;
        if (!nq) return;
        P0();
        const int w = tid >> 5, lane = tid & 31;
        const int h0 = ES->sym.nHdrs;
        __syncthreads();
#pragma unroll 1
        for (int base = 0; base < nq; base += ENG_NW) {
            const int r = base + w;
            const bool mine = r < nq && h0 + r < MAXH;
            if (mine) recode_one(ES->sym.qRec[r], w, lane, h0 + r);
            __syncthreads();
            if (w == 0) {   // intern the staged tables one after the other (two requests may produce the same table)
#pragma unroll 1
                for (int k = 0; k < ENG_NW && base + k < nq; k++) {
                    if (h0 + base + k >= MAXH) { if (lane == 0) ES->sym.overflow = 1; continue; }
                    const int t = intern_tab_warp(k, lane);
                    if (lane == 0 && !ES->sym.overflow) {
                        RSlot& rs = ES->sym.rc[ES->sym.qRec[base + k]];
                        rs.tabid = (unsigned short)t; rs.hid = (unsigned short)(h0 + base + k); rs.payload = ES->recPay[k]; rs.state = ST_DONE;
                    }
                    __syncwarp();
                }
            }
            __syncthreads();
        }
        if (tid == 0) ES->sym.nHdrs = min(MAXH, h0 + nq);
        __syncthreads();
        PCOUNT(PR_RECODE, nq - 1);
        P1(PR_RECODE);
    }

    // ---- header mutators, one warp per request ------------------------------------------------------------------------
    // replaceRLERunsWithLiteralsIfSmaller (DeflateBlockHuffman.java:321-332): in[0..np) -> out, returns the new count;
    // *saved = bits saved under CL
    static __device__ __forceinline__ int replace_runs_warp(const uint16_t* in, int np, const uint8_t* CL, bool prune, uint16_t* out,
                                                           int* saved, int lane) {
        int base = 0, sv = 0;
#pragma unroll 1
        for (int c0 = 0; c0 < np; c0 += 32) {
            const int i = c0 + lane;
            const uint16_t p = i < np ? in[i] : 0;
            const int run = i < np ? pair_run(p) : 0;
            bool rep = false;
            if (run > 0) {
                const int size = pair_size(p, CL);
                const int b = CL[pair_val(p)];
                const int tot = b * run;
                rep = b >= 1 && (prune ? tot <= size : tot < size);
                if (rep) sv += size - tot;
            }
            const int cnt = i < np ? (rep ? run : 1) : 0;
            int incl = cnt;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, dd); if (lane >= dd) incl += y; }
            int o = base + incl - cnt;
            if (rep) { const int vv = pair_val(p); const uint16_t q = pair_pack(vv, 0, vv); for (int k = 0; k < cnt; k++) out[o++] = q; }
            else if (cnt) out[o] = p;
            base += __shfl_sync(0xffffffffu, incl, 31);
        }
#pragma unroll 1
        for (int dd = 16; dd > 0; dd >>= 1) sv += __shfl_xor_sync(0xffffffffu, sv, dd);
        *saved = sv;
        __syncwarp();
        return base;
    }

    __device__ __noinline__ void hdrop_one(int src, int op, int dst, int w, int lane) {
        unsigned char* wsb = ES->u.ws[w];
        uint16_t* in = reinterpret_cast<uint16_t*>(wsb);                  // 320
        uint16_t* out = reinterpret_cast<uint16_t*>(wsb + 640);           // 320
        uint32_t* f19 = reinterpret_cast<uint32_t*>(wsb + 1280);          // 19
        uint8_t* cl = wsb + 1360;                                          // 19 old
        uint8_t* cl2 = wsb + 1392;                                         // 19 new
        unsigned char* tw = wsb + 1424;
        const Hdr& hs = hdrs[src];
        Hdr& hd = hdrs[dst];
        const int np = hs.np;
#pragma unroll 1
        for (int k = lane; k < np; k += 32) in[k] = hs.pairs[k];
        if (lane < 19) { cl[lane] = hs.CL[lane]; f19[lane] = 0; }
        int ncl = hs.ncl, bits = hs.bits;
        __syncwarp();
        const uint16_t* pairs = in;
        int npo = np;
        if (op == HOP_OPT) {   // optimiseHeader (:471-476): trailing zero code-length trim, then runs -> literals
            const int n2 = trim_ncl(cl, ncl);
            bits -= 3 * (ncl - n2);
            ncl = n2;
            int saved;
            npo = replace_runs_warp(in, np, cl, false, out, &saved, lane);
            bits -= saved;
            pairs = out;
            if (lane < 19) cl2[lane] = cl[lane];
        } else {               // recodeHeader (:579-629), after replaceRLERuns(prune) for the LessRLE variant (:632-635)
            if (op == HOP_RECODE_LESS) {
                int saved;
                npo = replace_runs_warp(in, np, cl, true, out, &saved, lane);
                pairs = out;
            }
#pragma unroll 1
            for (int k = lane; k < npo; k += 32) atomicAdd(&f19[pair_sym(pairs[k])], 1u);
            __syncwarp();
            if (lane == 0) hdr_code_from_freq(f19, cl2, ncl, &ncl, &bits, tw);   // numCodelenLens is NOT reset (H8)
            ncl = __shfl_sync(0xffffffffu, ncl, 0);
            bits = __shfl_sync(0xffffffffu, bits, 0);
        }
        __syncwarp();
#pragma unroll 1
        for (int k = lane; k < npo; k += 32) hd.pairs[k] = pairs[k];
        if (lane < 19) hd.CL[lane] = cl2[lane];
        if (lane == 0) { hd.np = (uint16_t)npo; hd.ncl = (uint8_t)ncl; hd.bits = bits; ES->sym.hbits[dst] = (unsigned short)bits; }
        __syncwarp();
    }

    __device__ __noinline__ void exec_hdrops() {
        const int nq = ES->sym.nqHdr;
        if (!nq) return;
        P0();
        const int w = tid >> 5, lane = tid & 31;
        const int h0 = ES->sym.nHdrs;
        __syncthreads();
#pragma unroll 1
        for (int r = w; r < nq; r += ENG_NW) {
            const int src = ES->sym.qHdr[r] >> 2, op = ES->sym.qHdr[r] & 3;
            if (h0 + r >= MAXH) { if (lane == 0) ES->sym.overflow = 1; continue; }
            hdrop_one(src, op, h0 + r, w, lane);
            if (lane == 0) ES->sym.hop[src][op] = (unsigned short)(h0 + r + 1);
        }
        __syncthreads();
        if (tid == 0) ES->sym.nHdrs = min(MAXH, h0 + nq);
        __syncthreads();
        PCOUNT(PR_HDROP, nq - 1);
        P1(PR_HDROP);
    }

    // ---- the 56 header strategy trials of the queued tables ----------------------------------------------------------
    // TRIAL_GROUP tables at a time: a warp cuts each table into runs (shared memory), then 28 threads per table evaluate
    // one rewrite strategy each for both prune values; the two header-code trees of a thread run in its own 100 bytes of
    // shared memory (huff_tree_tiny; the full algorithm in local memory only when a tree is deeper than 7)
#ifdef D4_TRIAL_GROUP
    static constexpr int TRIAL_GROUP = D4_TRIAL_GROUP;
#else
    static constexpr int TRIAL_GROUP = (ENG_NT / 28) < 6 ? (ENG_NT / 28) : 6;
#endif
    static constexpr int TRIAL_RL = 964, TRIAL_WS0 = ((TRIAL_GROUP * TRIAL_RL + 127) / 128) * 128;
    static_assert(TRIAL_WS0 + TRIAL_GROUP * 28 * TINY_WS_BYTES <= ENG_NW * WS_BYTES && TRIAL_WS0 + TRIAL_GROUP * 640 <= ENG_NW * WS_BYTES,
                  "trial workspaces fit the shared union");
    __device__ __noinline__ void exec_trials() {
        const int nq = ES->sym.nqTrial;
        if (!nq) return;
        P0();
        const int w = tid >> 5, lane = tid & 31;
        unsigned char* ub = &ES->u.ws[0][0];
#pragma unroll 1
        for (int base = 0; base < nq; base += TRIAL_GROUP) {
            const int cnt = nq - base < TRIAL_GROUP ? nq - base : TRIAL_GROUP;
            if (w < cnt)
                runlist_warp(tabs[ES->sym.qTrial[base + w]], *reinterpret_cast<RunList*>(ub + w * TRIAL_RL),
                             reinterpret_cast<uint16_t*>(ub + TRIAL_WS0 + w * 640), lane);
            __syncthreads();
            if (tid < cnt * 28) {
                const int b = tid / 28, c = tid % 28;
                const int t = ES->sym.qTrial[base + b];
                // c_trial_flags order: [0,20) and [40,48) are the rewrite strategies without prune, +20 / +8 with it
                const int kF = c < 20 ? c : 40 + (c - 20), kT = c < 20 ? 20 + c : 48 + (c - 20);
                TreeWsCLc slow;
                unsigned char* tw = ub + TRIAL_WS0 + tid * TINY_WS_BYTES;
                TreeWsTiny ws{reinterpret_cast<uint16_t*>(tw), tw + 48, &slow};
                int a = 0, bp = 0;
                if (trial_sizes(*reinterpret_cast<RunList*>(ub + b * TRIAL_RL), c_trial_flags[kF], &a, &bp, ws)) ES->err = ERR_TREE;
                trialAll[t * 56 + kF] = a;
                trialAll[t * 56 + kT] = bp;
            }
            __syncthreads();
            if (tid < cnt) {
                const int t = ES->sym.qTrial[base + tid];
                int best = 0x7fffffff, arg = 0;
#pragma unroll 1
                for (int k = 0; k < 56; k++) { const int bts = trialAll[t * 56 + k]; if (bts < best) { best = bts; arg = k; } }
                ES->sym.trialBits[t] = (unsigned short)best; ES->sym.trialArg[t] = (unsigned char)arg; ES->sym.trialState[t] = ST_DONE;
            }
            __syncthreads();
        }
        PCOUNT(PR_TRIALS, nq - 1);
        P1(PR_TRIALS);
    }

    __device__ __noinline__ void collect_recodes() {
        __syncthreads();
        if (tid == 0) ES->sym.nqRec = 0;
        __syncthreads();
#pragma unroll 1
        for (int k = tid; k < ES->sym.nMasks; k += ENG_NT)
            if (ES->sym.rc[k].state == ST_PENDING) {
                const int i = atomicAdd(&ES->sym.nqRec, 1);
                if (i < QREC) ES->sym.qRec[i] = (unsigned short)k;
            }
        __syncthreads();
        if (tid == 0) ES->sym.nqRec = min(ES->sym.nqRec, QREC);
        __syncthreads();
    }

    // the PENDING entries of the memo tables -> this step's request lists
    __device__ __noinline__ void collect_requests() {
        __syncthreads();
        if (tid == 0) { ES->sym.nqPass = ES->sym.nqRec = ES->sym.nqHdr = ES->sym.nqTrial = 0; }
        __syncthreads();
#pragma unroll 1
        for (int k = tid; k < PMEMO; k += ENG_NT)
            if (ES->sym.pm[k].key != 0 && ES->sym.pm[k].state != ST_DONE) {
                const int i = atomicAdd(&ES->sym.nqPass, 1);
                if (i < QPASS) ES->sym.qPass[i] = (unsigned short)k;
            }
#pragma unroll 1
        for (int k = tid; k < ES->sym.nHdrs * 3; k += ENG_NT)
            if (ES->sym.hop[k / 3][k % 3] == 0xFFFF) {
                const int i = atomicAdd(&ES->sym.nqHdr, 1);
                if (i < QHDR) ES->sym.qHdr[i] = (unsigned short)(((k / 3) << 2) | (k % 3));
            }
#pragma unroll 1
        for (int k = tid; k < ES->sym.nTabs; k += ENG_NT)
            if (ES->sym.trialState[k] == ST_PENDING) {
                const int i = atomicAdd(&ES->sym.nqTrial, 1);
                if (i < QTRIAL) ES->sym.qTrial[i] = (unsigned short)k;
            }
        __syncthreads();
        if (tid == 0) {   // what did not fit stays PENDING and is picked up by the next step
            ES->sym.nqPass = min(ES->sym.nqPass, QPASS);
            ES->sym.nqHdr = min(ES->sym.nqHdr, QHDR); ES->sym.nqTrial = min(ES->sym.nqTrial, QTRIAL);
        }
        collect_recodes();
    }

    // everything the last sweeps asked for.  Header trials feed nothing but the selection, so they wait until a batch
    // is worth the threads (or nothing else is left to do).
    __device__ __noinline__ void execute() {
        __syncthreads();
        exec_passes();
        collect_recodes();   // includes what the pruning passes of this step have just asked for
        exec_recodes();
        exec_hdrops();
        const bool others = ES->sym.nqPass + ES->sym.nqRec + ES->sym.nqHdr > 0;
        const bool doTrials = ES->sym.nqTrial && (!others || ES->sym.nqTrial >= 2 * TRIAL_GROUP);
        __syncthreads();
        if (doTrials) exec_trials();
        __syncthreads();
    }

    // ---- materialisation --------------------------------------------------------------------------------------------
    // candidate c (with header strategy `arg` when it is a trial winner) -> recs[which] + mask / histogram slot
    __device__ __noinline__ void materialise(const SC c, int arg, int which) {
        P0();
        __syncthreads();
        Cand& dst = recs[which];
        const int slot = which == 0 ? SLOT_B : SLOT_BEST;
        if (c.mid != slot) {
            const uint32_t* ms = maskp(c.mid);
            uint32_t* md = maskp(slot);
#pragma unroll 1
            for (uint32_t k = tid; k < v.nwords; k += ENG_NT) md[k] = ms[k];
            const uint32_t* hs = histp(c.mid);
            uint32_t* hd = histp(slot);
#pragma unroll 1
            for (int k = tid; k < 320; k += ENG_NT) hd[k] = hs[k];
        }
        const uint32_t* ts = (const uint32_t*)&tabs[c.tabid];
        uint32_t* td = (uint32_t*)&dst.tab;
        uint32_t* tm = (uint32_t*)&ES->u.mat.tab;
#pragma unroll 1
        for (int k = tid; k < (int)(sizeof(Tab) / 4); k += ENG_NT) { const uint32_t x = ts[k]; td[k] = x; tm[k] = x; }
        __syncthreads();
        if (c.type == 2) {
            if (arg >= 0) {   // a header strategy trial won: optimiseBlockDynBlock (DeflateStream.java:184-198) for real
                if (tid == 0) {
                    if (hdr_trial(ES->u.mat.tab, c_trial_flags[arg], ES->u.mat.hdr, ES->u.mat.ws)) ES->err = ERR_TREE;
                }
                __syncthreads();
                const uint32_t* hs = (const uint32_t*)&ES->u.mat.hdr;
                uint32_t* hd = (uint32_t*)&dst.hdr;
#pragma unroll 1
                for (int k = tid; k < (int)(sizeof(Hdr) / 4); k += ENG_NT) hd[k] = hs[k];
            } else {
                const uint32_t* hs = (const uint32_t*)&hdrs[c.hid];
                uint32_t* hd = (uint32_t*)&dst.hdr;
#pragma unroll 1
                for (int k = tid; k < (int)(sizeof(Hdr) / 4); k += ENG_NT) hd[k] = hs[k];
            }
        } else if (tid == 0) { dst.hdr.np = 0; dst.hdr.ncl = 0; dst.hdr.bits = 0; }
        if (tid == 0) { dst.payload = c.payload; dst.mid = 0; dst.tabid = 0; dst.pad2 = 0; }
        __syncthreads();
        P1(PR_MATERIAL);
    }

    // ---- one optimiseBlock call ---------------------------------------------------------------------------------------
    // sweeps + execution until the part `seg` of the enumeration is resolved, then the selection sweep.  Returns false on
    // a pool overflow (nothing selected).
    __device__ __noinline__ bool run_segment(unsigned seg) {
        if (tid == 0) { ES->sym.doneItem = 0; ES->sym.doneAor = 0; ES->itemNext = 0; }
        __syncthreads();
        // Lane 0 of every warp takes items (enum.cuh sweep_item) from a counter, each with its own copy of the enumerator.  The last
        // turn of the loop is the selection sweep: every item selects inside its own candidates (indices from 0, best so
        // far = the value carried in) into its record, and thread 0 joins the records in item order.  With the trace
        // armed the candidates must come out in order: thread 0 sweeps every item alone.
        bool selecting = false;
        const bool par = ES->en.trace == nullptr;
#pragma unroll 1
        for (int it = 0;; it++) {
            P0();   // a sweep is timed from here to the barrier after it: the slowest sweeper, and the join
            const bool serial = selecting && !par;
            const unsigned before = ES->en.bestIndex;
            if ((tid & 31) == 0 && (!serial || tid == 0)) {
                Enumer& en = serial ? ES->en : ES->u.sw.w[tid >> 5];
                if (!serial) { en = ES->en; en.trace = nullptr; }
                const long long carried = ES->en.bestSize;
                int next = 0;
#pragma unroll 1
                while (true) {
                    const int item = serial ? next++ : atomicAdd(&ES->itemNext, 1);
                    if (item >= NITEMS) break;
                    if (selecting && !serial) en.begin_item(carried);
                    const bool ok = en.sweep_one(ES->sym, selecting, seg, item);   // the one call site of the (inlined) sweep
                    if (selecting) {
                        if (!ok || en.internalError) ES->err = ERR_INTERNAL;
                        if (!serial) en.put_item(ES->u.sw.rec[item]);
                    }
                }
            }
            __syncthreads();
            if (tid == 0) ES->itemNext = 0;   // read again only after the barriers of collect_requests
            if (selecting) {
                if (tid == 0) ES->segImproved = par ? (ES->en.join(ES->u.sw.rec) ? 1 : 0) : (ES->en.bestIndex != before && !ES->en.bestStored);
                __syncthreads();
                P1(PR_SELECT);
                return true;
            }
            P1(PR_SWEEP);
            if (ES->sym.overflow) return false;
            collect_requests();
            const bool done = ES->sym.doneItem == (1u << NITEMS) - 1;
            const bool nothing = ES->sym.nqPass + ES->sym.nqRec + ES->sym.nqHdr + ES->sym.nqTrial == 0;
            if (done && nothing) { selecting = true; continue; }
            if (nothing || it > 4096) { if (tid == 0) ES->err = ERR_INTERNAL; __syncthreads(); return false; }
            execute();
            if (ES->sym.overflow) return false;
        }
    }

    // DeflateStream.optimiseBlock (:343-490) for B.  storedSize < 0: no stored candidate is compared (phase A resolves
    // it afterwards from sizeI / sizeC1 / restMin).  Result: ES->en.bestSize / bestStored / sizeI / sizeC1 / restMin /
    // bestIndex, and the winning Huffman candidate (B itself when nothing is smaller) materialised in recs[1].
    __device__ __noinline__ void optimise_block(long long storedSize) {
        P0();
        __syncthreads();
        if (tid == 0) { ES->en.storedSize = storedSize; ES->en.begin_round(ES->sym); ES->segmentedRound = 0; }
        __syncthreads();
        bool ok = run_segment(Enumer::SEG_ALL);
        if (ok) {
            materialise(ES->en.best, ES->en.bestArg, 1);
        } else if (!ES->err) {
            // a pool filled up: the same round again in four segments, with the pools reset (and B re-adopted) in between;
            // the running best lives in recs[1]
            PCOUNT(PR_SEGMENTED, 1);
            materialise(ES->en.B, -1, 0);
            __syncthreads();
            if (tid == 0) { ES->en.begin_round(ES->sym); ES->segmentedRound = 1; }   // the winner's ids belong to pools that are gone
            __syncthreads();
            const unsigned segs[4] = {Enumer::SEG_HEAD | Enumer::SEG_MULTI_H, Enumer::SEG_MULTI_O, Enumer::SEG_FIXED | Enumer::SEG_LEAST0,
                                      Enumer::SEG_LEAST1};
            bool haveBest = false;
#pragma unroll 1
            for (int k = 0; k < 4; k++) {
                const long long bs = ES->en.bestSize;
                const unsigned bi = ES->en.bestIndex, ci = ES->en.candIndex;
                const int bst = ES->en.bestStored;
                const long long rm = ES->en.restMin, c1 = ES->en.sizeC1;
                __syncthreads();
                adopt_B(false);
                if (tid == 0) {   // adopt_B rewrote B's ids; the selection state carries over
                    ES->en.bestSize = bs; ES->en.bestIndex = bi; ES->en.candIndex = ci; ES->en.bestStored = bst;
                    ES->en.restMin = rm; ES->en.sizeC1 = c1;
                }
                __syncthreads();
                if (!run_segment(segs[k])) { if (tid == 0 && !ES->err) ES->err = ERR_POOL; __syncthreads(); break; }
                if (ES->segImproved) { materialise(ES->en.best, ES->en.bestArg, 1); haveBest = true; }
                __syncthreads();
            }
            if (!haveBest && !ES->err) { adopt_B(false); materialise(ES->en.B, -1, 1); }
        }
        __syncthreads();
        P1(PR_ROUND);
    }

    // the winner of the last round becomes B (DeflateStream.java:514-530): pools and memo tables are kept while there is
    // room, since the next round revisits most of this round's states
    __device__ __noinline__ void advance_to_best() {
        P0();
        __syncthreads();
        const bool keep = !ES->segmentedRound && !ES->sym.overflow && ES->sym.nMasks <= MAXM / 2 && ES->sym.nTabs <= MAXT / 2 && ES->sym.nHdrs + 1 <= MAXH / 2 &&
                          ES->sym.nP <= PMEMO * 3 / 8 && ES->en.bestIndex != 0xffffffffu;
        // recs[0] := recs[1], slot B := slot BEST
        {
            const uint32_t* s = (const uint32_t*)&recs[1];
            uint32_t* d = (uint32_t*)&recs[0];
#pragma unroll 1
            for (int k = tid; k < (int)(sizeof(Cand) / 4); k += ENG_NT) d[k] = s[k];
            const uint32_t* ms = maskp(SLOT_BEST);
            uint32_t* md = maskp(SLOT_B);
#pragma unroll 1
            for (uint32_t k = tid; k < v.nwords; k += ENG_NT) md[k] = ms[k];
            const uint32_t* hs = histp(SLOT_BEST);
            uint32_t* hd = histp(SLOT_B);
#pragma unroll 1
            for (int k = tid; k < 320; k += ENG_NT) hd[k] = hs[k];
        }
        __syncthreads();
        if (keep) {
            SC b = ES->en.best;
            if (b.type == 2 && ES->en.bestArg >= 0) {   // the trial header only exists in the record: give it an id
                const int hid = ES->sym.nHdrs;
                const uint32_t* hs = (const uint32_t*)&recs[0].hdr;
                uint32_t* hd = (uint32_t*)&hdrs[hid];
#pragma unroll 1
                for (int k = tid; k < (int)(sizeof(Hdr) / 4); k += ENG_NT) hd[k] = hs[k];
                __syncthreads();
                if (tid == 0) {
                    ES->sym.hbits[hid] = (unsigned short)recs[0].hdr.bits;
                    ES->sym.nHdrs = hid + 1;
                    ES->sym.hop[hid][0] = ES->sym.hop[hid][1] = ES->sym.hop[hid][2] = 0;
                }
                b.hid = (short)hid;
            }
            __syncthreads();
            if (tid == 0) { ES->en.B = b; ES->en.blockType = b.type; }
            __syncthreads();
        } else {
            adopt_B(false);
        }
        P1(PR_REBASE);
    }
};

__device__ inline void eng_init(Eng& e, const EngScratch& sc, int cta) {
    e.tid = (int)threadIdx.x;
    e.maxwords = sc.maxwords;
    e.maxn = sc.maxwords * 32;
    unsigned char* base = sc.slab + (size_t)cta * sc.stride;
    e.masks = reinterpret_cast<uint32_t*>(base + sc.oMasks);
    e.tabs = reinterpret_cast<Tab*>(base + sc.oTabs);
    e.hdrs = reinterpret_cast<Hdr*>(base + sc.oHdrs);
    e.hists = reinterpret_cast<uint32_t*>(base + sc.oHists);
    e.tabHash = reinterpret_cast<unsigned long long*>(base + sc.oTabHash);
    e.dc = reinterpret_cast<short*>(base + sc.oDc);
    e.minfo = reinterpret_cast<uint32_t*>(base + sc.oMinfo);
    e.mout = reinterpret_cast<uint32_t*>(base + sc.oMout);
    e.mflag = reinterpret_cast<uint32_t*>(base + sc.oMflag);
    e.mrank = reinterpret_cast<uint32_t*>(base + sc.oMrank);
    e.litHist = reinterpret_cast<uint32_t*>(base + sc.oLitHist);
    e.tileFirst = reinterpret_cast<uint32_t*>(base + sc.oTileFirst);
    e.trialAll = reinterpret_cast<int*>(base + sc.oTrialAll);
    e.recs = reinterpret_cast<Cand*>(base + sc.oRecs);
    e.slowWs = reinterpret_cast<TreeWs<290, 584>*>(base + sc.oSlowWs);
    e.perm = reinterpret_cast<uint32_t*>(base + sc.oPerm);
    e.dcBits = reinterpret_cast<uint32_t*>(base + sc.oDcBits);
    e.items = reinterpret_cast<uint32_t*>(base + sc.oItems);
    e.bigWeights = false;
    if (threadIdx.x == 0) ES->err = 0;
    __syncthreads();
}

}  // namespace d4
