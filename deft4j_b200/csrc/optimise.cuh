// optimise.cuh — stream-level drivers around the candidate engine.
//
//   k_init_state : BlockRec (as parsed) -> BlkState (current model), one thread per block.
//   k_opt_blocks : phase A — DeflateStream.optimise's per-block fix-point loop (DeflateStream.java:504-530)
//                  for every block in parallel.  Huffman candidate sizes do not depend on the bit
//                  position, only the stored-block candidate does (DeflateBlockUncompressed.java:70-74),
//                  so each round logs (incumbent, "optimised" candidate, best of the rest) and
//                  k_finish replays the rounds with the real position to decide stored-vs-Huffman.
//   k_finish     : one CTA per stream — replays phase A with `pos` (incl. the reference's position
//                  drift, SURVEY.md H5, and the loop exit after an empty-block removal, H6), runs the
//                  merge phase (DeflateStream.mergeBlocks, :568-650) sequentially with the engine, and
//                  lays the final blocks out (bit positions, BFINAL, stream size, bits saved).
#pragma once
#include "engine.cuh"

namespace d4 {

constexpr int MAXR = 64;  // optimiseBlock rounds logged per block

struct BlkState {
    Cand cand;            // cand.tab.type: 0 STORED, 1 FIXED, 2 DYNAMIC
    uint64_t sym_off;     // symbol pool index
    uint64_t out_off;     // decoded pool offset
    uint64_t mask_off;    // word offset in the mask pool
    uint64_t out_len;
    uint32_t n_sym;
    int32_t alive;
    int32_t bfinal;
    int32_t nrounds;
    uint64_t bit_pos;     // position of the 3-bit header in the rewritten stream
    long long size_bits;  // getSizeBits(bit_pos + 3)
};
struct RoundRec { long long sizeI, sizeC1, restMin, best; };   // one optimiseBlock round of phase A
struct RoundLog { RoundRec r[MAXR]; };

struct StreamState {
    uint64_t blk_base;
    uint32_t n_blocks;
    uint32_t cut;          // blocks [0, cut) take part in phase A (first removable empty block index)
    uint32_t selected;     // 0: leave untouched (not part of this optimise call)
    int32_t status;
    long long saved_bits;
    uint64_t total_bits;   // getSizeBits() of the current model
};

__device__ __forceinline__ long long stored_size(uint64_t len, long long alignment) {
    long long c = alignment % 8;
    c = c == 0 ? 0 : 8 - c;
    return ((long long)len + 4) * 8 + c;
}
__device__ __forceinline__ long long blk_size(const BlkState& b, long long alignment) {
    return b.cand.tab.type == 0 ? stored_size(b.out_len, alignment) : cand_size(b.cand);
}

__global__ void k_init_state(const BlockRec* __restrict__ recs, const uint64_t* __restrict__ mask_offs,
                             BlkState* __restrict__ bs, uint64_t nblk) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nblk) return;
    const BlockRec& r = recs[i];
    BlkState& b = bs[i];
    b.cand.tab = r.tab;
    b.cand.tab.type = r.type;
    b.cand.tab.pad[0] = b.cand.tab.pad[1] = b.cand.tab.pad[2] = 0;
    b.cand.hdr = r.hdr;
    b.cand.payload = r.payload_bits;
    b.sym_off = r.sym_base;   // pool indices (rebased by k_compact_blocks)
    b.out_off = r.out_base;
    b.mask_off = mask_offs[i];
    b.out_len = r.out_len;
    b.n_sym = r.n_sym;
    b.alive = 1;
    b.bfinal = r.bfinal;
    b.nrounds = 0;
    b.bit_pos = r.hdr_bit;
    b.size_bits = (long long)(r.end_bit - r.hdr_bit) - 3;
}

// the view of block b for the engine
__device__ inline void eng_view(Eng& e, const BlkState& b, const uint32_t* sym, const uint32_t* symout, const uint8_t* out,
                                uint32_t n, uint64_t ulen) {
    e.v.sym = sym + b.sym_off;
    e.v.symout = symout + b.sym_off;
    e.v.out = out;
    e.v.n = n;
    e.v.nm = 0;       // (load_block counts the matches)
    e.v.nwords = 0;
    e.v.ulen = ulen;
    e.v.out_off = b.out_off;
}

// --------------------------------------------------------------------------------------------------
// phase A
// --------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(ENG_NT, D4_ENG_MINB)
k_opt_blocks(const uint32_t* __restrict__ jobs, uint32_t njobs, BlkState* __restrict__ bs, RoundLog* __restrict__ logs,
             const uint32_t* __restrict__ sym, const uint32_t* __restrict__ symout, const uint8_t* __restrict__ out,
             uint32_t* __restrict__ maskpool, EngScratch sc, unsigned* __restrict__ counter, int* __restrict__ gerr) {
    EngSmem& S = g_es;
    __shared__ uint32_t s_job;
    Eng e;
    eng_init(e, sc, blockIdx.x);
    const int tid = threadIdx.x;
    while (true) {
        if (tid == 0) s_job = atomicAdd(counter, 1u);
        __syncthreads();
        const uint32_t job = s_job;
        __syncthreads();
        if (job >= njobs) break;
        P0();
        BlkState& b = bs[jobs[job]];
        eng_view(e, b, sym, symout, out, b.n_sym, b.out_len);
        e.load_block(b.cand, maskpool + b.mask_off, false);   // zeros after parse; the current symbol list on a repeated call
        RoundLog& lg = logs[jobs[job]];
        int r = 0;
        long long prevBest = -1;
        while (true) {
            e.optimise_block(-1);
            if (S.err) break;
            if (tid == 0 && r < MAXR) {
                RoundRec rr; rr.sizeI = S.en.sizeI; rr.sizeC1 = S.en.sizeC1; rr.restMin = S.en.restMin; rr.best = S.en.bestSize;
                lg.r[r] = rr;
            }
            // self-checks: this round's incumbent is the previous round's winner; the winner's payload recomputed from
            // its symbol list; a winning header trial sized exactly as the size-only evaluation said
            const bool improved = S.en.bestSize < S.en.sizeI;
            bool bad = prevBest >= 0 && S.en.sizeI != prevBest;
            int badWhat = 1;
            __syncthreads();
            if (improved) {
                e.pass_hist_full(SLOT_BEST);
                const long long truePay = e.hist_payload(S.hist, e.recs[1].tab);
                if (truePay != e.recs[1].payload) { bad = true; badWhat = 2; }
                if (cand_size(e.recs[1]) != S.en.bestSize) { bad = true; badWhat = 3; }
            }
            if (bad && tid == 0) {
                if (atomicMax(gerr, 13) < 13) {
                    gerr[1] = (int)jobs[job]; gerr[2] = r; gerr[3] = (int)S.en.bestIndex;
                    gerr[4] = (int)S.en.bestSize; gerr[5] = (int)cand_size(e.recs[1]); gerr[6] = badWhat; gerr[7] = (int)prevBest;
                }
            }
            __syncthreads();
            prevBest = S.en.bestSize;
            r++;
            if (!improved) break;
            if (r >= MAXR) { if (tid == 0) S.err = ERR_ROUNDS; break; }
            e.advance_to_best();
        }
        __syncthreads();
        // write the fix-point back: recs[0] / slot B hold it once a round has improved (the last round never does)
        if (r > 1 && !S.err) {
            const uint32_t* s = (const uint32_t*)&e.recs[0];
            uint32_t* d = (uint32_t*)&b.cand;
            for (int k = tid; k < (int)(sizeof(Cand) / 4); k += ENG_NT) d[k] = s[k];
            e.store_mask(SLOT_B, maskpool + b.mask_off);
        }
        if (tid == 0) b.nrounds = r;
        __syncthreads();
        if (S.err) { if (tid == 0) { atomicMax(gerr, S.err); S.err = 0; } }
        __syncthreads();
        P1(PR_BLOCK);
    }
}

// --------------------------------------------------------------------------------------------------
// k_finish: replay + merge + layout, one CTA per stream
// --------------------------------------------------------------------------------------------------
__device__ void finish_stream(EngSmem& S, Eng& e, StreamState& st, BlkState* __restrict__ bs, const RoundLog* __restrict__ logs,
                              uint32_t* __restrict__ sym, const uint32_t* __restrict__ symout, const uint8_t* __restrict__ out,
                              uint32_t* __restrict__ maskpool, int merge, int* __restrict__ gerr) {
    __shared__ long long s_pos, s_saved;
    __shared__ int s_cur, s_next, s_do, s_first;
    if (!st.selected || st.status != ST_OK) return;
    const int tid = threadIdx.x;
    BlkState* B = bs + st.blk_base;
    const uint32_t nb = st.n_blocks;

    // ---- replay of DeflateStream.optimise (:496-566) with the real bit position --------------------
    // The walk is sequential in `pos` (one thread), so the CTA stages what it reads — block type, decoded length and
    // the first rounds of the log — in shared memory a tile of blocks at a time (the engine's shared state is not
    // live yet); the serial loop then never waits on global memory.
    {
        constexpr int RT = 64, RR = 4;   // blocks per tile, rounds staged per block
        struct Tile { unsigned long long out_len[RT]; int type[RT]; RoundRec rr[RT][RR]; };
        static_assert(sizeof(Tile) <= sizeof(EngSmem), "replay tile must fit in the engine's shared storage");
        Tile& T = *reinterpret_cast<Tile*>(&S);
        __shared__ long long s_rpos, s_rsaved;
        __shared__ int s_stop;
        __shared__ uint32_t s_first_alive, s_n_alive;
        if (tid == 0) { s_rpos = 0; s_rsaved = 0; s_stop = 0; s_first_alive = nb; s_n_alive = 0; }
        __syncthreads();
        {   // first live block and their number: every thread looks at its share (one thread walking all the block
            // states paid a global-memory round trip per block)
            uint32_t fa = nb, na = 0;
            for (uint32_t k = tid; k < nb; k += ENG_NT) if (B[k].alive) { if (fa == nb) fa = k; na++; }
            if (na) { atomicMin(&s_first_alive, fa); atomicAdd(&s_n_alive, na); }
        }
        __syncthreads();
        const uint32_t first_alive = s_first_alive, n_alive = s_n_alive;
        for (uint32_t t0 = 0; t0 < nb && !s_stop; t0 += RT) {
            const uint32_t cnt = nb - t0 < RT ? nb - t0 : RT;
            for (uint32_t k = tid; k < cnt; k += ENG_NT) {
                T.out_len[k] = B[t0 + k].out_len;
                T.type[k] = B[t0 + k].alive ? (int)B[t0 + k].cand.tab.type : -1;   // -1: removed by an earlier optimise call
            }
            for (uint32_t q = tid; q < cnt * RR; q += ENG_NT) T.rr[q / RR][q % RR] = logs[st.blk_base + t0 + q / RR].r[q % RR];
            __syncthreads();
            if (tid == 0) {
                long long pos = s_rpos, saved = s_rsaved;
                for (uint32_t kk = 0; kk < cnt; kk++) {
                    const uint32_t k = t0 + kk;
                    const unsigned long long out_len = T.out_len[kk];
                    if (T.type[kk] < 0) continue;
                    if (out_len > 0 || (k == first_alive && n_alive == 1)) {
                        if (T.type[kk] == 0) {  // stored blocks have no candidates
                            pos += 3;
                            pos += stored_size(out_len, pos);
                        } else {
                            const RoundLog& lg = logs[st.blk_base + k];
                            int r = 0;
                            while (true) {
                                pos += 3;
                                const RoundRec rr = r < RR ? T.rr[kk][r] : lg.r[r];
                                const long long I = rr.sizeI, C1 = rr.sizeC1, R = rr.restMin, W = rr.best;
                                const long long m1 = I < C1 ? I : C1;
                                bool storedWins = false;
                                long long Ssz = 0;
                                if (out_len <= 65535) {
                                    Ssz = stored_size(out_len, pos);
                                    storedWins = Ssz < m1 && Ssz <= R;
                                }
                                if (storedWins) {
                                    saved += I - Ssz;
                                    B[k].cand.tab.type = 0;
                                    pos += stored_size(out_len, pos);
                                    // next pass over the (now stored) block finds nothing
                                    pos += 3;
                                    pos += stored_size(out_len, pos);
                                    break;
                                }
                                if (W < I) { saved += I - W; pos += W; r++; continue; }
                                pos += I;
                                break;
                            }
                        }
                    } else {  // empty block: removed, and the reference's loop ends here (H6)
                        saved += blk_size(B[k], pos + 3) + 3;
                        B[k].alive = 0;
                        // its EOB (an empty Huffman block is one symbol) must not surface inside a later merge of its
                        // neighbours, whose symbol range spans it (DeflateBlockHuffman.merge, :1233-1271)
                        if (B[k].cand.tab.type != 0 && B[k].n_sym) sym[B[k].sym_off + B[k].n_sym - 1] = SYM_NOP;
                        s_stop = 1;
                        break;
                    }
                }
                s_rpos = pos; s_rsaved = saved;
            }
            __syncthreads();
        }
        if (tid == 0) { s_saved = s_rsaved; S.err = 0; }  // the tile overlaid the engine state: start it clean
    }
    __syncthreads();

    // ---- DeflateStream.mergeBlocks (:568-650) ---------------------------------------------------------
    if (merge) {
        if (tid == 0) {
            s_pos = 0; s_first = 1;
            int c = 0;
            while (c < (int)nb && !B[c].alive) c++;
            s_cur = c;
        }
        __syncthreads();
        while (true) {
            const int cur = s_cur;
            if (cur >= (int)nb) break;
            if (tid == 0) {
                int n = cur + 1;
                while (n < (int)nb && !B[n].alive) n++;
                s_next = n < (int)nb ? n : -1;
                s_do = 0;
                BlkState& c = B[cur];
                if (s_first && s_next < 0) {
                    s_pos += blk_size(c, s_pos + 3) + 3;
                    s_do = 3;  // advance
                } else if (c.out_len > 0) {
                    s_pos += 3;
                    if (s_next >= 0) {
                        BlkState& nx = B[s_next];
                        if (c.cand.tab.type == 0) {
                            if (c.out_len + nx.out_len <= 65535) {  // stored + anything, by size only
                                long long curSize = blk_size(c, s_pos);
                                long long nextSize = blk_size(nx, s_pos + curSize + 3);
                                long long mergedSize = stored_size(c.out_len + nx.out_len, s_pos);
                                long long cs = curSize + 3 + nextSize - mergedSize;
                                if (cs > 0) {
                                    s_saved += cs;
                                    c.out_len += nx.out_len;
                                    c.n_sym = 0;
                                    nx.alive = 0;
                                    s_do = 2;  // merged: same block again
                                }
                            }
                        } else if (nx.cand.tab.type != 0) {
                            s_do = 1;  // Huffman + Huffman: needs the engine
                        }
                    }
                    if (s_do == 0) s_do = 3;
                    if (s_do != 1) s_pos += blk_size(c, s_pos);
                } else {
                    s_saved += blk_size(c, s_pos + 3) + 3;
                    c.alive = 0;
                    s_do = 4;  // removed: loop ends (H6)
                }
            }
            __syncthreads();
            int action = s_do;
            if (action == 1) {
                BlkState& c = B[cur];
                BlkState& nx = B[s_next];
                const uint32_t nA = c.n_sym, nB = nx.n_sym;
                // merged symbol list = A without its EOB + B (DeflateBlockHuffman.merge, :1233-1271).  A removed empty
                // Huffman block may sit between the two in the pool (its EOB is a NOP by now), so B's symbols start
                // `gap` symbols after A's first one, not nA.
                const uint32_t gap = (uint32_t)(nx.sym_off - c.sym_off), span = gap + nB;
                if (tid == 0) sym[c.sym_off + nA - 1] = SYM_NOP;
                eng_view(e, c, sym, symout, out, span, c.out_len + nx.out_len);
                // the merged mask is assembled in the pool region of A, which has room for the union (the regions of A, a
                // removed block in between and B are adjacent); B's own region is left alone until the merge is accepted
                {
                    uint32_t* m = e.maskp(SLOT_BEST);   // symbol-space scratch until the round materialises its winner
                    for (uint32_t k = tid; k < e.sym_words(); k += ENG_NT) m[k] = 0;
                    __syncthreads();
                    const uint32_t* ma = maskpool + c.mask_off;
                    const uint32_t* mb = maskpool + nx.mask_off;
                    for (uint32_t i = tid; i < nA; i += ENG_NT)
                        if ((ma[i >> 5] >> (i & 31)) & 1) atomicOr(&m[i >> 5], 1u << (i & 31));
                    for (uint32_t i = tid; i < nB; i += ENG_NT)
                        if ((mb[i >> 5] >> (i & 31)) & 1) atomicOr(&m[(gap + i) >> 5], 1u << ((gap + i) & 31));
                    __syncthreads();
                    // both halves recoded to the fixed code; payload from the histogram (DeflateBlockHuffman.merge)
                    e.load_block(c.cand, m, true);
                }
                const long long pos = s_pos;
                e.optimise_block(stored_size(e.v.ulen, pos));
                if (tid == 0) {
                    long long curSize = blk_size(c, pos);
                    long long nextSize = blk_size(nx, pos + curSize + 3);
                    long long cs = curSize + 3 + nextSize - S.en.bestSize;
                    s_do = cs > 0 ? 5 : 6;
                    if (cs > 0) s_saved += cs;
                }
                __syncthreads();
                if (s_do == 5) {  // accept
                    if (!S.en.bestStored) {
                        const uint32_t* s = (const uint32_t*)&e.recs[1];
                        uint32_t* d = (uint32_t*)&c.cand;
                        for (int k = tid; k < (int)(sizeof(Cand) / 4); k += ENG_NT) d[k] = s[k];
                        e.store_mask(SLOT_BEST, maskpool + c.mask_off);
                    }
                    __syncthreads();
                    if (tid == 0) {
                        if (S.en.bestStored) c.cand.tab.type = 0;
                        c.n_sym = span;
                        c.out_len += nx.out_len;
                        nx.alive = 0;
                    }
                } else {
                    if (tid == 0) sym[c.sym_off + nA - 1] = 256;  // restore the EOB
                }
                __syncthreads();
                if (tid == 0) s_pos += blk_size(c, s_pos);
                action = (s_do == 5) ? 2 : 3;
                __syncthreads();
            }
            if (action == 4) break;
            if (tid == 0) {
                if (action == 3) {  // finishPass
                    s_cur = s_next < 0 ? (int)nb : s_next;
                    s_first = 0;
                }
            }
            __syncthreads();
        }
        if (S.err && tid == 0) { atomicMax(gerr, S.err); S.err = 0; }
    }
    __syncthreads();

    // ---- layout: DeflateStream.getSizeBits (:171-182) + BFINAL from list position (:128-145) ----------
    // sequential in the running size; inputs and outputs are staged through shared memory like the replay above
    {
        constexpr int LT = 128;
        struct LTile { unsigned long long out_len[LT], bit_pos[LT]; long long csize[LT], size_bits[LT]; int type[LT], alive[LT]; };
        static_assert(sizeof(LTile) <= sizeof(EngSmem), "layout tile must fit in the engine's shared storage");
        __syncthreads();
        LTile& T = *reinterpret_cast<LTile*>(&S);
        __shared__ long long s_size;
        __shared__ int s_last;
        if (tid == 0) { s_size = 0; s_last = -1; }
        __syncthreads();
        for (uint32_t t0 = 0; t0 < nb; t0 += LT) {
            const uint32_t cnt = nb - t0 < LT ? nb - t0 : LT;
            for (uint32_t k = tid; k < cnt; k += ENG_NT) {
                const BlkState& b = B[t0 + k];
                T.out_len[k] = b.out_len; T.type[k] = b.cand.tab.type; T.alive[k] = b.alive; T.csize[k] = cand_size(b.cand);
            }
            __syncthreads();
            if (tid == 0) {
                long long size = s_size;
                int last = s_last;
                for (uint32_t k = 0; k < cnt; k++) {
                    if (!T.alive[k]) continue;
                    T.bit_pos[k] = (unsigned long long)size;
                    size += 3;
                    T.size_bits[k] = T.type[k] == 0 ? stored_size(T.out_len[k], size) : T.csize[k];
                    size += T.size_bits[k];
                    last = (int)(t0 + k);
                }
                s_size = size; s_last = last;
            }
            __syncthreads();
            for (uint32_t k = tid; k < cnt; k += ENG_NT) {
                if (!T.alive[k]) continue;
                BlkState& b = B[t0 + k];
                b.bit_pos = T.bit_pos[k]; b.size_bits = T.size_bits[k]; b.bfinal = 0;
            }
            __syncthreads();
        }
        if (tid == 0) {
            if (s_last >= 0) B[s_last].bfinal = 1;
            st.total_bits = (uint64_t)s_size;
            st.saved_bits = s_saved;
        }
        __syncthreads();
    }
}

// streams are taken from a queue by a grid sized to the machine, so the engine scratch is per CTA, not per stream
__global__ void __launch_bounds__(ENG_NT, D4_ENG_MINB)
k_finish(StreamState* __restrict__ streams, uint32_t nstreams, BlkState* __restrict__ bs, const RoundLog* __restrict__ logs,
         uint32_t* __restrict__ sym, const uint32_t* __restrict__ symout, const uint8_t* __restrict__ out,
         uint32_t* __restrict__ maskpool, EngScratch sc, int merge, unsigned* __restrict__ counter, int* __restrict__ gerr) {
    EngSmem& S = g_es;
    __shared__ uint32_t s_job;
    Eng e;
    if (merge) eng_init(e, sc, blockIdx.x);
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) s_job = atomicAdd(counter, 1u);
        __syncthreads();
        const uint32_t job = s_job;
        if (job >= nstreams) break;
        finish_stream(S, e, streams[job], bs, logs, sym, symout, out, maskpool, merge, gerr);
    }
}

}  // namespace d4
