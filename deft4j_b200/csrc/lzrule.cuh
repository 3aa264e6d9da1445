// lzrule.cuh — the parse rule of the device compressor (deft4cu_compress_batch), shared by the kernels (lzcomp.cuh) and
// the host restatement in hosttest.cu, so the CPU suite pins the very code the kernels run.
//
// The output is a pure function of the input bytes and the block size B:
//   blocks     : B input bytes each, the last one shorter; an empty stream is one block holding only EOB.
//   hash       : h(p) = ((d[p] << 10) ^ (d[p+1] << 5) ^ d[p+2]) & 0x7FFF for p + 3 <= N (zlib's 15-bit hash);
//                the last two bytes of a stream have no hash and are never candidates.
//   candidates : the LZ_CHAIN most recent q < p with h(q) == h(p) and p - q <= LZ_WINDOW, newest first; entries whose
//                bytes do not match still count.  The window may reach into earlier blocks, never before the stream.
//   match at p : common prefix of d[q..] and d[p..], capped at min(258, e - p) (a match never leaves its block).  The
//                longest wins, the newest on ties.  Length < 3 is no match, and so is length 3 at a distance > 4096.
//   lazy parse : from i = s: take M(i) when it exists and (i + 1 == e or M(i+1).len <= M(i).len), else the literal d[i];
//                then EOB.  Every block is FIXED, only the last has BFINAL, length 258 is always symbol 285.
#pragma once
#include "common.cuh"

namespace d4 {

constexpr uint32_t LZ_WINDOW = 32768, LZ_CHAIN = 32, LZ_MAX_LEN = 258, LZ_TOO_FAR = 4096, LZ_HASH_MASK = 0x7FFF;
constexpr uint32_t LZ_BLOCK_DEFAULT = 32768, LZ_BLOCK_MIN = 256, LZ_BLOCK_MAX = 65535;

__host__ __device__ inline uint32_t lz_hash(uint32_t a, uint32_t b, uint32_t c) { return ((a << 10) ^ (b << 5) ^ c) & LZ_HASH_MASK; }

// M(p) packed as len << 16 | dist (0: no match)
__host__ __device__ inline uint32_t lz_pack(uint32_t len, uint32_t dist) { return (len << 16) | dist; }
__host__ __device__ inline uint32_t lz_mlen(uint32_t m) { return m >> 16; }
__host__ __device__ inline uint32_t lz_mdist(uint32_t m) { return m & 0xFFFFu; }

// length symbol (257..285) of a match length 3..258; 258 is always 285
__host__ __device__ inline int lz_len_sym(int len) {
    if (len == 258) return 285;
    const unsigned l = (unsigned)len - 3;
    if (l < 8) return 257 + (int)l;
#ifdef __CUDA_ARCH__
    const int hb = 31 - __clz(l);
#else
    const int hb = 31 - __builtin_clz(l);
#endif
    return 257 + 4 * (hb - 1) + (int)((l >> (hb - 2)) & 3);
}
// bits of a symbol under the fixed code (RFC 1951 3.2.6)
__host__ __device__ inline int lz_fixed_lit_bits(int byte) { return byte <= 143 ? 8 : 9; }
__host__ __device__ inline int lz_fixed_match_bits(int len, int dist) {
    const int ls = lz_len_sym(len), ds = dist_sym(dist);
    return (ls <= 279 ? 7 : 8) + len_ebits_of(ls) + 5 + dist_ebits_of(ds);
}
constexpr int LZ_FIXED_EOB_BITS = 7;

// M(p) for p in block [s, e) of a stream.  `byte(i)` reads stream byte i; `prev(q)` is the next older chain entry of q
// (the most recent q' < q with h(q') == h(q)) or -1.  Both are called only inside [p - LZ_WINDOW, e + 2).
template <class Byte, class Prev>
__host__ __device__ inline uint32_t lz_best_match(int64_t p, int64_t e, int64_t N, Byte byte, Prev prev) {
    if (p + 3 > N) return 0;
    const int64_t cap64 = e - p < (int64_t)LZ_MAX_LEN ? e - p : (int64_t)LZ_MAX_LEN;
    const uint32_t cap = (uint32_t)cap64;
    if (cap < 3) return 0;
    uint32_t best = 0, bestd = 0;
    int64_t q = prev(p);
    for (uint32_t k = 0; k < LZ_CHAIN && q >= 0 && p - q <= (int64_t)LZ_WINDOW; k++) {
        uint32_t l = 0;
        while (l < cap && byte(q + l) == byte(p + l)) l++;
        if (l > best) { best = l; bestd = (uint32_t)(p - q); if (l == cap) break; }
        q = prev(q);
    }
    if (best < 3 || (best == 3 && bestd > LZ_TOO_FAR)) return 0;
    return lz_pack(best, bestd);
}

// the lazy step at i (block end e): the match to emit there, or 0 for the literal
__host__ __device__ inline uint32_t lz_take(uint32_t mi, uint32_t mnext, bool last) {
    if (!mi) return 0;
    return (last || lz_mlen(mnext) <= lz_mlen(mi)) ? mi : 0;
}

}  // namespace d4
