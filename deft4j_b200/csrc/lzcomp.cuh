// lzcomp.cuh — the device compressor: raw bytes -> the model parse() builds for a FIXED-coded stream (BlockRecs, sym /
// symout, decoded bytes), so that the candidate engine does the entropy coding exactly as for a parsed fixed stream.
// The parse rule is lzrule.cuh.
//
//   k_lz_match : one CTA per block (persistent, jobs from a counter).  The block's window d[max(0, s - 32 K), min(N, e + 2))
//                is staged in shared memory next to a 32 K-entry head table.  Warp 0 links every window position to the
//                previous one with the same hash, 32 positions per step (__match_any_sync finds the closest lower lane
//                with the same hash; the highest lane of each group moves the head); the links go to the CTA's slab in
//                global memory (u16 distances, L2 resident).  Then every thread finds M(p) for its positions of [s, e),
//                takes the lazy decision, and the CTA walks the parse in 512 chunks with the same self-synchronising
//                fix-up k_count uses (a chunk re-walks from where its predecessor really ended until nothing changes).
//                A scan over the chunks gives each chunk's first symbol and the block's symbol count and payload bits.
//   k_lz_emit  : one CTA per block, after the host has placed every block's symbols in the pool: each thread re-walks
//                its chunk writing sym / symout, thread 0 writes EOB and the FIXED BlockRec.
#pragma once
#include "lzrule.cuh"
#include "parse.cuh"

namespace d4 {

constexpr int LZ_NT = 512;
constexpr uint32_t LZ_WIN_CAP = ((LZ_WINDOW + LZ_BLOCK_MAX + 2) + 15) & ~15u;    // staged window bytes (and slab links)
constexpr uint32_t LZ_SMEM = LZ_WIN_CAP + (LZ_HASH_MASK + 1) * 4;                  // window + head table (229 392 B)

struct LzJob {
    uint64_t base;       // pool offset of the stream's first byte
    uint64_t n;          // stream length
    uint32_t s, e;       // the block: stream bytes [s, e)
    uint64_t sym_base;   // pool index of the block's first symbol (set by the host before k_lz_emit)
    uint64_t hdr_bit;    // stream-relative bit position of the block header (same)
    uint32_t bfinal, pad;
};
struct LzRes { uint32_t n_sym, payload; };

__global__ void __launch_bounds__(LZ_NT, 1)
k_lz_match(const LzJob* __restrict__ jobs, uint32_t njobs, const uint8_t* __restrict__ out, uint32_t* __restrict__ M,
           uint16_t* __restrict__ slab, uint2* __restrict__ ent, LzRes* __restrict__ res, unsigned* __restrict__ counter) {
    extern __shared__ __align__(16) uint8_t s_dyn[];
    uint8_t* win = s_dyn;
    uint32_t* head = (uint32_t*)(s_dyn + LZ_WIN_CAP);
    uint16_t* step = (uint16_t*)head;   // after the links are built: step | fixed bits << 9 per block position
    __shared__ uint32_t s_exit[LZ_NT];
    __shared__ uint32_t s_wc[LZ_NT / 32], s_wb[LZ_NT / 32];
    __shared__ uint32_t s_job;
    uint16_t* link = slab + (size_t)blockIdx.x * LZ_WIN_CAP;
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    while (true) {
        if (t == 0) s_job = atomicAdd(counter, 1u);
        __syncthreads();
        const uint32_t j = s_job;
        if (j >= njobs) break;
        const LzJob jb = jobs[j];
        const int64_t s = jb.s, e = jb.e, N = (int64_t)jb.n;
        const int64_t w0 = s > (int64_t)LZ_WINDOW ? s - (int64_t)LZ_WINDOW : 0;
        const int64_t wend = e + 2 < N ? e + 2 : N;
        const uint32_t wlen = (uint32_t)(wend - w0);
        const uint8_t* src = out + jb.base + w0;
        for (uint32_t i = t; i < wlen; i += LZ_NT) win[i] = src[i];
        for (uint32_t i = t; i <= LZ_HASH_MASK; i += LZ_NT) head[i] = 0xFFFFFFFFu;
        __syncthreads();
        // ---- hash chains of the window (warp 0, 32 positions a step) ------------------------------------------------
        const int64_t hend = (e < N - 2 ? e : N - 2) - w0;   // window positions with a hash that a match of [s, e) can reach
        if (wid == 0 && hend > 0) {
            for (uint32_t c = 0; c < (uint32_t)hend; c += 32) {
                const uint32_t r = c + lane;
                const bool valid = r < (uint32_t)hend;
                const uint32_t h = valid ? lz_hash(win[r], win[r + 1], win[r + 2]) : 0x10000u + lane;
                const uint32_t grp = __match_any_sync(0xFFFFFFFFu, h);
                const uint32_t lower = grp & ((1u << lane) - 1u);
                uint32_t q = 0xFFFFFFFFu;
                if (valid) q = lower ? c + (31 - __clz(lower)) : head[h];
                __syncwarp();
                if (valid && (grp >> lane) == 1u) head[h] = r;
                if (valid) link[r] = (q != 0xFFFFFFFFu && r - q <= LZ_WINDOW) ? (uint16_t)(r - q) : (uint16_t)0;
                __syncwarp();
            }
        }
        __syncthreads();
        // ---- M(p) for the block's positions --------------------------------------------------------------------------
        const uint32_t L = (uint32_t)(e - s);
        auto byte = [&](int64_t i) { return win[i - w0]; };
        auto prev = [&](int64_t q) -> int64_t { const uint32_t d = link[q - w0]; return d ? q - d : -1; };
        uint32_t* Mb = M + jb.base + s;
        for (uint32_t i = t; i < L; i += LZ_NT) {
            const uint32_t m = lz_best_match(s + i, e, N, byte, prev);
            Mb[i] = m;
            step[i] = (uint16_t)lz_mlen(m);
        }
        __syncthreads();
        // lazy decision: M keeps the match taken at i, 0 where a literal is emitted
        for (uint32_t i = t; i < L; i += LZ_NT) Mb[i] = lz_take(Mb[i], lz_pack(i + 1 < L ? step[i + 1] : 0u, 0), i + 1 == L);
        __syncthreads();
        for (uint32_t i = t; i < L; i += LZ_NT) {
            const uint32_t m = Mb[i];
            step[i] = m ? (uint16_t)(lz_mlen(m) | (lz_fixed_match_bits((int)lz_mlen(m), (int)lz_mdist(m)) << 9))
                        : (uint16_t)(1u | (lz_fixed_lit_bits(win[s - w0 + i]) << 9));
        }
        __syncthreads();
        // ---- the parse: chunks of C positions, each walked from where its predecessor ended ------------------------
        const uint32_t C = (L + LZ_NT - 1) / LZ_NT;
        const uint32_t a = min((uint32_t)t * C, L), b = min((uint32_t)(t + 1) * C, L);
        uint32_t entry = a, cnt = 0, bits = 0, exitp = a;
        bool need = true, changed;
        do {
            if (need) {
                uint32_t p = entry;
                cnt = 0; bits = 0;
                while (p < b) { const uint32_t v = step[p]; p += v & 511u; bits += v >> 9; cnt++; }
                exitp = p;
                s_exit[t] = exitp;
            }
            __syncthreads();
            need = false;
            if (t > 0 && s_exit[t - 1] != entry) { entry = s_exit[t - 1]; need = true; }
            changed = __syncthreads_or(need);
        } while (changed);
        // ---- exclusive scan of the chunks' symbol counts and bits -----------------------------------------------------
        uint32_t ci = cnt, bi = bits;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, ci, d), y = __shfl_up_sync(0xFFFFFFFFu, bi, d);
            if (lane >= d) { ci += x; bi += y; }
        }
        if (lane == 31) { s_wc[wid] = ci; s_wb[wid] = bi; }
        __syncthreads();
        if (wid == 0) {
            const uint32_t x0 = lane < LZ_NT / 32 ? s_wc[lane] : 0u, y0 = lane < LZ_NT / 32 ? s_wb[lane] : 0u;
            uint32_t x = x0, y = y0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, x, d), v = __shfl_up_sync(0xFFFFFFFFu, y, d);
                if (lane >= d) { x += u; y += v; }
            }
            if (lane < LZ_NT / 32) { s_wc[lane] = x - x0; s_wb[lane] = y - y0; }
            if (lane == LZ_NT / 32 - 1) res[j] = LzRes{x + 1, y + (uint32_t)LZ_FIXED_EOB_BITS};   // + EOB
        }
        __syncthreads();
        ent[(size_t)j * LZ_NT + t] = make_uint2(entry, s_wc[wid] + ci - cnt);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(LZ_NT)
k_lz_emit(const LzJob* __restrict__ jobs, const uint8_t* __restrict__ out, const uint32_t* __restrict__ M,
          const uint2* __restrict__ ent, const LzRes* __restrict__ res, uint32_t* __restrict__ sym, uint32_t* __restrict__ symout,
          BlockRec* __restrict__ blocks) {
    const uint32_t j = blockIdx.x;
    const LzJob jb = jobs[j];
    const int t = threadIdx.x;
    const uint32_t L = jb.e - jb.s;
    const uint32_t C = (L + LZ_NT - 1) / LZ_NT;
    const uint32_t b = min((uint32_t)(t + 1) * C, L);
    const uint2 en = ent[(size_t)j * LZ_NT + t];
    const uint64_t ob = jb.base + jb.s;
    const uint32_t* Mb = M + ob;
    uint64_t k = jb.sym_base + en.y;
    for (uint32_t p = en.x; p < b; k++) {
        const uint32_t m = Mb[p];
        if (m) {
            const int len = (int)lz_mlen(m);
            sym[k] = sym_pack_match(len, (int)lz_mdist(m), 0, lz_len_sym(len));
            symout[k] = (uint32_t)(ob + p);
            p += len;
        } else {
            sym[k] = out[ob + p];
            symout[k] = (uint32_t)(ob + p);
            p++;
        }
    }
    // the record as k_count / k_emit leave it for a FIXED block
    uint32_t* rw = (uint32_t*)&blocks[j];
    for (int w = t; w < (int)(sizeof(BlockRec) / 4); w += LZ_NT) rw[w] = 0;
    __syncthreads();
    if (t == 0) {
        const LzRes r = res[j];
        sym[jb.sym_base + r.n_sym - 1] = 256;
        symout[jb.sym_base + r.n_sym - 1] = (uint32_t)(ob + L);
        BlockRec& br = blocks[j];
        br.hdr_bit = jb.hdr_bit;
        br.data_bit = jb.hdr_bit + 3;
        br.end_bit = jb.hdr_bit + 3 + r.payload;
        br.sym_base = jb.sym_base;
        br.out_base = ob;
        br.n_sym = r.n_sym;
        br.out_len = L;
        br.payload_bits = r.payload;
        br.type = 1;
        br.bfinal = (uint8_t)jb.bfinal;
        fixed_lens(br.tab.L, br.tab.D);
        br.tab.nL = 286; br.tab.nD = 30; br.tab.type = 1;
    }
}

}  // namespace d4
