// deft4cu.cu — host side of libdeft4cu.so: the C ABI of include/deft4cu.h on top of the kernels in
// parse.cuh / engine.cuh / optimise.cuh / write.cuh.  Host code only moves bytes and sizes buffers; all
// deflate work (decode, LZ77, cost model, enumeration, bit writing) is in the kernels.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <chrono>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/deft4cu.h"

namespace d4 {
static thread_local std::string g_err;
static void set_error(const std::string& s) { g_err = s; }
}  // namespace d4

#include "write.cuh"
#include "checksum.cuh"
#include "lzcomp.cuh"

namespace d4 {

static int g_device = -1;
static int g_sms = 148;
static bool g_sync_debug = getenv("D4_SYNC") != nullptr;
static uint64_t g_opt_launches = 0;   // launches of the candidate engine (k_opt_blocks) since start: tests count them
static std::mutex g_mu;

// D4_HOST_TIMING=1: wall time of the host-side phases on stderr (diagnostics for the container path)
struct HostTimer {
    const char* what; std::chrono::steady_clock::time_point t0; bool on;
    explicit HostTimer(const char* w) : what(w), t0(std::chrono::steady_clock::now()) { static bool e = getenv("D4_HOST_TIMING") != nullptr; on = e; }
    ~HostTimer() {
        if (on && g_device >= 0) {
            cudaMemPool_t pool;
            uint64_t res = 0, used = 0;
            if (cudaDeviceGetDefaultMemPool(&pool, g_device) == cudaSuccess) {
                cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &res);
                cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
            }
            fprintf(stderr, "[deft4cu] pool reserved %7.1f MiB used %7.1f MiB  ", res / 1048576.0, used / 1048576.0);
        }
        if (on) fprintf(stderr, "[deft4cu] %-14s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    }
};

static int ensure_init() {
    if (g_device >= 0) return DEFT4CU_OK;
    return deft4cu_init(0);
}

#define LAUNCH(kern, grid, block, stream, ...)                                   \
    do {                                                                         \
        kern<<<(grid), (block), 0, (stream)>>>(__VA_ARGS__);                     \
        launches++;                                                              \
        D4_CUDA_CHECK(cudaGetLastError());                                       \
        if (g_sync_debug) {                                                      \
            cudaError_t se_ = cudaStreamSynchronize(stream);                     \
            if (se_ != cudaSuccess) {                                            \
                set_error(std::string(#kern) + " faulted: " + cudaGetErrorString(se_)); \
                return DEFT4CU_ERR_CUDA;                                         \
            }                                                                    \
        }                                                                        \
    } while (0)

// the same with dynamic shared memory (opt-in above 48 KiB is set once in deft4cu_init)
#define LAUNCH_SM(kern, grid, block, smem, stream, ...)                          \
    do {                                                                         \
        kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);                \
        launches++;                                                              \
        D4_CUDA_CHECK(cudaGetLastError());                                       \
        if (g_sync_debug) {                                                      \
            cudaError_t se_ = cudaStreamSynchronize(stream);                     \
            if (se_ != cudaSuccess) {                                            \
                set_error(std::string(#kern) + " faulted: " + cudaGetErrorString(se_)); \
                return DEFT4CU_ERR_CUDA;                                         \
            }                                                                    \
        }                                                                        \
    } while (0)

template <typename T>
static cudaError_t dalloc(T** p, size_t n, cudaStream_t s) {
    *p = nullptr;
    if (n == 0) n = 1;
    return cudaMallocAsync((void**)p, n * sizeof(T), s);
}
template <typename T>
static void dfree(T*& p, cudaStream_t s) {
    if (p) cudaFreeAsync((void*)p, s);
    p = nullptr;
}

// parity-debug trace buffer (deft4cu_debug_trace_*): while armed, phase A runs the blocks one after the other in
// stream order on a single CTA, so that the log reads like the reference's sequential optimise loop
static long long* g_trace_dev = nullptr;
static uint32_t g_trace_dev_cap = 0;

struct BlkSummary { uint32_t type, n_sym; uint64_t out_len; uint32_t alive, pad; };

// Result buffers handed to the caller (deft4cu_result::out) live in pinned host blocks so that the device -> host
// copy of a batch's output is one DMA at PCIe speed; blocks are reference counted by the `out` pointers that point
// into them and recycled by deft4cu_free_results / deft4cu_free_buffer (pinning memory is slow, so a few idle blocks
// are kept).
struct HostBlock { uint8_t* p; size_t cap; int refs; bool pinned; };
static std::mutex g_hmu;
static std::vector<HostBlock> g_hblocks;
static uint8_t* host_block_acquire(size_t bytes, int refs) {
    std::lock_guard<std::mutex> lk(g_hmu);
    int best = -1;
    for (size_t k = 0; k < g_hblocks.size(); k++)
        if (g_hblocks[k].refs == 0 && g_hblocks[k].cap >= bytes && (best < 0 || g_hblocks[k].cap < g_hblocks[best].cap)) best = (int)k;
    if (best < 0) {
        // drop idle blocks that are too small before growing
        for (size_t k = 0; k < g_hblocks.size();) {
            if (g_hblocks[k].refs == 0) {
                if (g_hblocks[k].pinned) cudaFreeHost(g_hblocks[k].p); else free(g_hblocks[k].p);
                g_hblocks.erase(g_hblocks.begin() + k);
            } else k++;
        }
        HostBlock hb{nullptr, (bytes + (1u << 20)) & ~(size_t)((1u << 20) - 1), 0, true};
        if (cudaMallocHost((void**)&hb.p, hb.cap) != cudaSuccess) {
            cudaGetLastError();
            hb.pinned = false;
            hb.p = (uint8_t*)malloc(hb.cap);
            if (!hb.p) return nullptr;
        }
        g_hblocks.push_back(hb);
        best = (int)g_hblocks.size() - 1;
    }
    g_hblocks[best].refs = refs;
    return g_hblocks[best].p;
}
static void host_release(const uint8_t* ptr) {
    if (!ptr) return;
    std::lock_guard<std::mutex> lk(g_hmu);
    for (auto& hb : g_hblocks)
        if (ptr >= hb.p && ptr < hb.p + hb.cap) { if (hb.refs > 0) hb.refs--; return; }
}

__global__ void k_blk_summary(const BlockRec* __restrict__ recs, BlkSummary* __restrict__ out, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i].type = recs[i].type;
    out[i].n_sym = recs[i].n_sym;
    out[i].out_len = recs[i].out_len;
    out[i].alive = 1; out[i].pad = 0;
}
// the same from the current model: a second optimise call on a batch sees merged / removed / stored blocks
__global__ void k_state_summary(const BlkState* __restrict__ bs, BlkSummary* __restrict__ out, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i].type = bs[i].cand.tab.type;
    out[i].n_sym = bs[i].n_sym;
    out[i].out_len = bs[i].out_len;
    out[i].alive = bs[i].alive ? 1u : 0u; out[i].pad = 0;
}

class Batch {
   public:
    uint32_t n = 0;
    cudaStream_t cs = nullptr;      // stream every kernel and copy of this batch is issued on
    cudaStream_t own_cs = nullptr;  // created by upload(); cs may later be redirected to a caller's stream
    uint64_t launches = 0;
    float ms[8] = {0};

    std::vector<uint64_t> in_len, in_off;
    uint64_t total_in = 0;
    uint8_t* d_in = nullptr;

    std::vector<StreamDesc> descs;
    std::vector<StreamInfo> infos;
    StreamDesc* d_descs = nullptr;
    StreamInfo* d_infos = nullptr;
    BlockRec* d_blocks = nullptr;
    ChunkRec* d_chunks = nullptr;
    uint64_t nblk_total = 0, nsym_total = 0, nout_total = 0;
    uint32_t* d_sym = nullptr;
    uint32_t* d_symout = nullptr;
    uint8_t* d_out = nullptr;

    std::vector<BlkSummary> summ;
    std::vector<uint32_t> blk_stream;
    std::vector<uint64_t> mask_offs;
    uint64_t maskwords_total = 0;
    uint32_t* d_blk_stream = nullptr;
    BlkState* d_bs = nullptr;
    RoundLog* d_logs = nullptr;
    uint32_t* d_maskpool = nullptr;
    std::vector<StreamState> sstate;
    StreamState* d_sstate = nullptr;
    int* d_gerr = nullptr;
    std::vector<int64_t> size_bits_in;

    uint8_t* d_dst = nullptr;
    std::vector<uint8_t> h_dst;   // host copy of d_dst, filled by the first per-stream write of a multi-stream batch
    std::vector<uint64_t> dst_off, dst_len;
    uint64_t dst_total = 0;
    uint64_t* d_dst_off = nullptr;
    std::vector<uint32_t> crc, adler;
    bool have_sums = false;
    bool parsed = false;
    bool optimised = false;
    bool too_big = false;   // parse() refused: the decoded size of the batch does not fit the 32-bit pools (split it)
    bool compressed = false;   // the model was built by compress() from raw bytes (the input must never be parsed)
    uint32_t block_bytes = 0;  // compress(): input bytes per block

    ~Batch() { release_all(); if (own_cs) cudaStreamDestroy(own_cs); }

    void release_model() {
        dfree(d_descs, cs); dfree(d_infos, cs); dfree(d_blocks, cs); dfree(d_chunks, cs);
        dfree(d_sym, cs); dfree(d_symout, cs); dfree(d_out, cs);
        dfree(d_blk_stream, cs); dfree(d_bs, cs); dfree(d_logs, cs); dfree(d_maskpool, cs);
        dfree(d_sstate, cs); dfree(d_gerr, cs); dfree(d_dst, cs); dfree(d_dst_off, cs);
        parsed = false; compressed = false; have_sums = false; optimised = false;
    }
    void release_all() {
        HostTimer ht("release");
        drop_stage();
        release_model();
        dfree(d_in, cs);
        if (cs) cudaStreamSynchronize(cs);
    }

    int upload(const uint8_t* const* in, const uint64_t* len, uint32_t count) {
        HostTimer ht("upload");
        n = count;
        if (!own_cs) { D4_CUDA_CHECK(cudaStreamCreateWithFlags(&own_cs, cudaStreamNonBlocking)); cs = own_cs; }
        in_len.assign(len, len + n);
        in_off.resize(n);
        uint64_t off = 0;
        for (uint32_t i = 0; i < n; i++) { in_off[i] = off; off += (in_len[i] + 32 + 15) & ~15ull; }
        total_in = off + 512;   // k_find loads three 8-byte words per thread of its last tile (FIND_TILE / 8 + 24 bytes)
        D4_CUDA_CHECK(dalloc(&d_in, total_in, cs));
        // Many small streams (a folder of PNGs, the entries of a ZIP): a copy per stream from pageable memory costs ~10 us
        // each, so they are gathered by a few host threads into one pinned block and go over in a single DMA.
        if (n >= 16 && total_in <= (1ull << 30) && !getenv("D4_NO_STAGING")) {
            stage = host_block_acquire(total_in, 1);
            if (stage) {
                auto fill = [&](uint32_t lo, uint32_t hi) {
                    for (uint32_t i = lo; i < hi; i++) {
                        if (in_len[i]) memcpy(stage + in_off[i], in[i], in_len[i]);
                        const uint64_t end = in_off[i] + in_len[i], nxt = i + 1 < n ? in_off[i + 1] : total_in;
                        memset(stage + end, 0, nxt - end);
                    }
                };
                const uint32_t nt = (uint32_t)std::min<uint64_t>(8, std::max<uint64_t>(1, total_in >> 22));
                if (nt <= 1) fill(0, n);
                else {
                    // equal shares of BYTES, cut at stream boundaries
                    std::vector<uint32_t> cut(nt + 1, n);
                    cut[0] = 0;
                    for (uint32_t t = 1, i = 0; t < nt; t++) {
                        while (i < n && in_off[i] < total_in / nt * t) i++;
                        cut[t] = i;
                    }
                    std::vector<std::thread> th;
                    for (uint32_t t = 1; t < nt; t++) th.emplace_back(fill, cut[t], cut[t + 1]);
                    fill(cut[0], cut[1]);
                    for (auto& x : th) x.join();
                }
                D4_CUDA_CHECK(cudaMemcpyAsync(d_in, stage, total_in, cudaMemcpyHostToDevice, cs));
                return DEFT4CU_OK;   // (the block goes back to the pool after parse()'s first synchronisation)
            }
        }
        D4_CUDA_CHECK(cudaMemsetAsync(d_in, 0, total_in, cs));
        for (uint32_t i = 0; i < n; i++)
            if (in_len[i]) D4_CUDA_CHECK(cudaMemcpyAsync(d_in + in_off[i], in[i], in_len[i], cudaMemcpyHostToDevice, cs));
        return DEFT4CU_OK;
    }
    uint8_t* stage = nullptr;   // pinned staging block of upload(), held until the copy has completed
    void drop_stage() {
        if (stage) { cudaStreamSynchronize(cs); host_release(stage); stage = nullptr; }
    }

    // the same from streams that already sit in other batches' input buffers (device to device)
    int upload_from(const std::vector<std::pair<Batch*, uint32_t>>& src) {
        n = (uint32_t)src.size();
        if (!own_cs) { D4_CUDA_CHECK(cudaStreamCreateWithFlags(&own_cs, cudaStreamNonBlocking)); cs = own_cs; }
        in_len.resize(n); in_off.resize(n);
        uint64_t off = 0;
        for (uint32_t i = 0; i < n; i++) { in_len[i] = src[i].first->in_len[src[i].second]; in_off[i] = off; off += (in_len[i] + 32 + 15) & ~15ull; }
        total_in = off + 512;
        D4_CUDA_CHECK(dalloc(&d_in, total_in, cs));
        D4_CUDA_CHECK(cudaMemsetAsync(d_in, 0, total_in, cs));
        for (uint32_t i = 0; i < n; i++) {
            Batch* b = src[i].first;
            D4_CUDA_CHECK(cudaStreamSynchronize(b->cs));   // its upload has finished
            if (in_len[i]) D4_CUDA_CHECK(cudaMemcpyAsync(d_in + in_off[i], b->d_in + b->in_off[src[i].second], in_len[i], cudaMemcpyDeviceToDevice, cs));
        }
        return DEFT4CU_OK;
    }

    // ---- parse: find block boundaries, count (walkers), emit, LZ77 resolve, model init ---------------------
    std::vector<StreamDesc> wdescs;     // per walker (device copy: d_descs)
    std::vector<StreamInfo> winfos;     // per walker
    std::vector<uint32_t> chain;        // valid walkers, stream after stream, in stream order
    std::vector<uint32_t> chain_off;    // n + 1 offsets into chain
    uint32_t parse_rewalks = 0, parse_walkers = 0;

    int parse() {
        HostTimer ht("parse");
        release_model();
        too_big = false;
        cudaEvent_t ev[4];
        for (auto& e : ev) cudaEventCreate(&e);
        descs.assign(n + 1, StreamDesc{});
        infos.assign(n, StreamInfo{});
        D4_CUDA_CHECK(dalloc(&d_gerr, 8, cs));
        D4_CUDA_CHECK(cudaMemsetAsync(d_gerr, 0, 8 * sizeof(int), cs));
        // ---- walkers: one per segment of each stream -------------------------------------------------------
        uint64_t seg_bytes = 128 << 10;
        if (const char* e = getenv("D4_SEG_BYTES")) seg_bytes = std::max<uint64_t>(64, strtoull(e, nullptr, 10));
        const uint64_t seg_bits = seg_bytes * 8;
        const uint64_t spec_max_bits = 4 * seg_bits + (1 << 20);
        wdescs.clear();
        std::vector<uint32_t> w0(n), spec_list, all_list;
        for (uint32_t i = 0; i < n; i++) {
            const uint32_t nseg = in_len[i] <= seg_bytes ? 1u : (uint32_t)((in_len[i] + seg_bytes - 1) / seg_bytes);
            w0[i] = (uint32_t)wdescs.size();
            for (uint32_t j = 0; j < nseg; j++) {
                StreamDesc d{};
                d.in_off = in_off[i]; d.in_len = in_len[i];
                d.start_bit = j == 0 ? 0 : BIT_NONE;
                d.stop_bit = nseg == 1 ? BIT_NONE : (uint64_t)(j + 1) * seg_bits;
                d.walker0 = w0[i]; d.nseg = nseg; d.spec = j == 0 ? 0 : 1;
                if (nseg == 1) { d.blk_cap = in_len[i] / 4096 + 8; d.chunk_cap = in_len[i] * 8 / CHUNK_BITS + d.blk_cap + 8; }
                else { d.blk_cap = seg_bytes / 2048 + 8; d.chunk_cap = 4 * seg_bits / CHUNK_BITS + d.blk_cap + 8; }
                if (j) spec_list.push_back((uint32_t)wdescs.size());
                all_list.push_back((uint32_t)wdescs.size());
                wdescs.push_back(d);
            }
        }
        const uint32_t W = (uint32_t)wdescs.size();
        parse_walkers = W; parse_rewalks = 0;
        std::vector<uint32_t> wstream(W);
        for (uint32_t i = 0; i < n; i++) for (uint32_t j = 0; j < wdescs[w0[i]].nseg; j++) wstream[w0[i] + j] = i;
        winfos.assign(W, StreamInfo{});
        uint32_t* d_list = nullptr;
        D4_CUDA_CHECK(dalloc(&d_descs, (size_t)W, cs));
        D4_CUDA_CHECK(dalloc(&d_infos, (size_t)W, cs));
        D4_CUDA_CHECK(dalloc(&d_list, (size_t)W, cs));
        cudaEventRecord(ev[0], cs);
        if (!spec_list.empty()) {
            D4_CUDA_CHECK(cudaMemcpyAsync(d_descs, wdescs.data(), sizeof(StreamDesc) * W, cudaMemcpyHostToDevice, cs));
            D4_CUDA_CHECK(cudaMemcpyAsync(d_list, spec_list.data(), 4 * spec_list.size(), cudaMemcpyHostToDevice, cs));
            LAUNCH(k_find, (unsigned)spec_list.size(), FIND_NT, cs, d_in, d_descs, d_list, seg_bits);
            // the candidate starts come back to the host: the chain below compares them with the true boundaries
            std::vector<StreamDesc> tmp(W);
            D4_CUDA_CHECK(cudaMemcpyAsync(tmp.data(), d_descs, sizeof(StreamDesc) * W, cudaMemcpyDeviceToHost, cs));
            D4_CUDA_CHECK(cudaStreamSynchronize(cs));
            for (uint32_t w : spec_list) wdescs[w].start_bit = tmp[w].start_bit;
        }
        chain.clear(); chain_off.assign(n + 1, 0);
        std::vector<std::vector<uint32_t>> chains(n);
        std::vector<uint8_t> trunc(n, 0);
        for (int attempt = 0;; attempt++) {
            uint64_t bt = 0, ct = 0;
            for (uint32_t w = 0; w < W; w++) {
                wdescs[w].blk_base = bt; bt += wdescs[w].blk_cap;
                wdescs[w].chunk_base = ct; ct += wdescs[w].chunk_cap;
            }
            dfree(d_blocks, cs); dfree(d_chunks, cs);
            D4_CUDA_CHECK(dalloc(&d_blocks, bt, cs));
            D4_CUDA_CHECK(dalloc(&d_chunks, ct, cs));
            D4_CUDA_CHECK(cudaMemcpyAsync(d_descs, wdescs.data(), sizeof(StreamDesc) * W, cudaMemcpyHostToDevice, cs));
            D4_CUDA_CHECK(cudaMemcpyAsync(d_list, all_list.data(), 4 * (size_t)W, cudaMemcpyHostToDevice, cs));
            if (W) LAUNCH_SM(k_count, W, PARSE_NT, WIN_BYTES + WIN_SLACK + 16, cs, d_in, d_descs, d_infos, d_blocks, d_chunks, d_list, seg_bits, spec_max_bits);
            D4_CUDA_CHECK(cudaMemcpyAsync(winfos.data(), d_infos, sizeof(StreamInfo) * W, cudaMemcpyDeviceToHost, cs));
            D4_CUDA_CHECK(cudaStreamSynchronize(cs));
            if (stage && cs == own_cs) { host_release(stage); stage = nullptr; }   // upload()'s copy is behind us
            // ---- follow every stream's chain from walker 0; re-walk what was guessed wrong ---------------------
            std::vector<uint32_t> cur(n), pending;
            std::vector<uint8_t> fin(n, 0);
            for (uint32_t i = 0; i < n; i++) { chains[i].assign(1, w0[i]); cur[i] = w0[i]; }
            bool overflow = false;
            while (true) {
                pending.clear();
                for (uint32_t i = 0; i < n; i++) {
                    if (fin[i]) continue;
                    while (true) {
                        const StreamInfo& wi = winfos[cur[i]];
                        const StreamDesc& wd = wdescs[cur[i]];
                        if (wi.n_blocks > wd.blk_cap || wi.n_chunks > wd.chunk_cap) { overflow = true; fin[i] = 1; break; }
                        if (wi.status != ST_OK || wi.final_seen) { fin[i] = 1; break; }
                        if (wi.end_bit + 3 > in_len[i] * 8) { fin[i] = 2; break; }  // no room for another block header (:81-84)
                        uint64_t j = wi.end_bit / seg_bits;
                        if (j >= wd.nseg) j = wd.nseg - 1;
                        const uint32_t nx = w0[i] + (uint32_t)j;
                        if (nx <= cur[i]) {  // cannot happen (a walker stops at or past its segment end); refuse rather than loop
                            set_error("parse chain did not advance");
                            return DEFT4CU_ERR_CUDA;
                        }
                        chains[i].push_back(nx);
                        cur[i] = nx;
                        if (wdescs[nx].start_bit == wi.end_bit && winfos[nx].status != ST_NONE && winfos[nx].status != ST_ABORT)
                            continue;  // guessed right
                        wdescs[nx].start_bit = wi.end_bit;
                        wdescs[nx].spec = 0;
                        pending.push_back(nx);
                        break;
                    }
                }
                if (pending.empty()) break;
                parse_rewalks += (uint32_t)pending.size();
                for (uint32_t w : pending)
                    D4_CUDA_CHECK(cudaMemcpyAsync(d_descs + w, &wdescs[w], sizeof(StreamDesc), cudaMemcpyHostToDevice, cs));
                D4_CUDA_CHECK(cudaMemcpyAsync(d_list, pending.data(), 4 * pending.size(), cudaMemcpyHostToDevice, cs));
                LAUNCH_SM(k_count, (unsigned)pending.size(), PARSE_NT, WIN_BYTES + WIN_SLACK + 16, cs, d_in, d_descs, d_infos, d_blocks, d_chunks, d_list, seg_bits, spec_max_bits);
                for (uint32_t w : pending)
                    D4_CUDA_CHECK(cudaMemcpyAsync(&winfos[w], d_infos + w, sizeof(StreamInfo), cudaMemcpyDeviceToHost, cs));
                D4_CUDA_CHECK(cudaStreamSynchronize(cs));
            }
            for (uint32_t i = 0; i < n; i++) trunc[i] = fin[i] == 2;
            if (!overflow) break;
            if (attempt == 3) { set_error("block/chunk capacity retry failed"); return DEFT4CU_ERR_CUDA; }
            // record slots ran out somewhere on a chain: size every walker that has run for what it reported (the
            // starts found so far are kept, so the next attempt follows the same chain without guessing again)
            for (uint32_t w = 0; w < W; w++) {
                if (winfos[w].status == ST_NONE) continue;
                wdescs[w].blk_cap = std::max<uint64_t>(wdescs[w].blk_cap, winfos[w].n_blocks + 8);
                wdescs[w].chunk_cap = std::max<uint64_t>(wdescs[w].chunk_cap, 2 * winfos[w].n_chunks + 8);
            }
        }
        // ---- per-stream totals -------------------------------------------------------------------------------
        for (uint32_t i = 0; i < n; i++) {
            StreamInfo& si = infos[i];
            si = StreamInfo{};
            si.status = ST_OK;
            for (uint32_t w : chains[i]) {
                const StreamInfo& wi = winfos[w];
                si.n_blocks += wi.n_blocks; si.n_syms += wi.n_syms; si.out_len += wi.out_len; si.n_chunks += wi.n_chunks;
                si.end_bit = wi.end_bit;
                if (wi.status != ST_OK) { si.status = wi.status >= ST_NONE ? ST_PARSE : wi.status; break; }
            }
            if (trunc[i] && si.status == ST_OK) si.status = ST_PARSE;
            if (si.out_len > 0xF0000000ull && si.status == ST_OK) si.status = ST_UNSUPPORTED;
            si.total_bits = si.end_bit;
            si.consumed = (si.end_bit + 7) >> 3;
            chain_off[i] = (uint32_t)chain.size();
            if (si.status == ST_OK) chain.insert(chain.end(), chains[i].begin(), chains[i].end());
        }
        chain_off[n] = (uint32_t)chain.size();
        dfree(d_list, cs);
        cudaEventRecord(ev[1], cs);
        // pool bases: streams back to back, inside a stream its valid walkers in chain order
        uint64_t sb = 0, ob = 0;
        for (uint32_t i = 0; i < n; i++) {
            descs[i].sym_base = sb; descs[i].out_base = ob;
            for (uint32_t c = chain_off[i]; c < chain_off[i + 1]; c++) {
                StreamDesc& wd = wdescs[chain[c]];
                wd.sym_base = sb; wd.out_base = ob; wd.stream_out_base = descs[i].out_base;
                sb += winfos[chain[c]].n_syms; ob += winfos[chain[c]].out_len;
            }
        }
        descs[n].sym_base = sb; descs[n].out_base = ob;
        nsym_total = sb; nout_total = ob;
        uint64_t ob_max = 0xF8000000ull;   // decoded offsets are 32-bit
        if (const char* e = getenv("D4_MAX_DECODED")) ob_max = std::min<uint64_t>(ob_max, strtoull(e, nullptr, 10));   // tests force the split
        if (ob >= ob_max) {
            too_big = true;
            for (uint32_t i = 0; i < n; i++) if (infos[i].status == ST_OK) infos[i].status = ST_UNSUPPORTED;
            set_error("decoded size of the batch exceeds 4 GiB; split the batch");
            return DEFT4CU_ERR_UNSUPPORTED;
        }
        D4_CUDA_CHECK(cudaMemcpyAsync(d_descs, wdescs.data(), sizeof(StreamDesc) * W, cudaMemcpyHostToDevice, cs));
        D4_CUDA_CHECK(dalloc(&d_sym, sb, cs));
        D4_CUDA_CHECK(dalloc(&d_symout, sb, cs));
        D4_CUDA_CHECK(dalloc(&d_out, ob + 16, cs));
        // block list (compact, in stream order)
        std::vector<EmitJob> jobs;
        blk_stream.clear();
        std::vector<uint64_t> sblk_base(n);
        for (uint32_t i = 0; i < n; i++) {
            sblk_base[i] = blk_stream.size();
            for (uint32_t c = chain_off[i]; c < chain_off[i + 1]; c++)
                for (uint32_t k = 0; k < winfos[chain[c]].n_blocks; k++) { jobs.push_back(EmitJob{chain[c], k}); blk_stream.push_back(i); }
        }
        nblk_total = jobs.size();
        EmitJob* d_jobs = nullptr;
        D4_CUDA_CHECK(dalloc(&d_jobs, jobs.size(), cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(EmitJob) * jobs.size(), cudaMemcpyHostToDevice, cs));
        if (!jobs.empty())
            LAUNCH(k_emit, (unsigned)jobs.size(), 256, cs, d_in, d_descs, d_blocks, d_chunks, d_jobs, d_infos, d_sym, d_symout, d_out);
        cudaEventRecord(ev[2], cs);
        // LZ77
        if (ob) {
            uint32_t* d_ptr = nullptr;
            int* d_changed = nullptr;
            uint8_t* d_done = nullptr;
            D4_CUDA_CHECK(dalloc(&d_ptr, ob, cs));
            D4_CUDA_CHECK(dalloc(&d_changed, 1, cs));
            D4_CUDA_CHECK(dalloc(&d_done, ob, cs));
            D4_CUDA_CHECK(cudaMemsetAsync(d_done, 0, ob, cs));
            if (sb) LAUNCH(k_lz_fill, (unsigned)((sb + 255) / 256), 256, cs, d_sym, d_symout, sb, d_out, d_ptr);
            // stored bytes are roots (k_emit wrote them into d_out; their pointers are set here)
            LAUNCH(k_lz_root_stored, (unsigned)std::max<uint64_t>(1, nblk_total), 256, cs, d_descs, d_blocks, d_jobs, (uint32_t)nblk_total, d_ptr);
            for (int it = 0; it < 64; it++) {
                int changed = 0;
                D4_CUDA_CHECK(cudaMemsetAsync(d_changed, 0, sizeof(int), cs));
                if (it == 0) {
                    uint32_t tile = LZJ_TILE;
                    if (const char* e = getenv("D4_LZ_TILE")) tile = (uint32_t)std::max(512, atoi(e)) / LZJ_NT * LZJ_NT;
                    LAUNCH(k_lz_jump_tiles, (unsigned)((ob + tile - 1) / tile), LZJ_NT, cs, d_ptr, d_out, d_done, ob, tile, d_changed);
                }
                else LAUNCH(k_lz_jump, (unsigned)((ob + 1023) / 1024), 256, cs, d_ptr, d_out, d_done, ob, d_changed);
                D4_CUDA_CHECK(cudaMemcpyAsync(&changed, d_changed, sizeof(int), cudaMemcpyDeviceToHost, cs));
                D4_CUDA_CHECK(cudaStreamSynchronize(cs));
                if (!changed) break;
                if (it == 63) { set_error("LZ77 resolve did not converge"); return DEFT4CU_ERR_CUDA; }
            }
            dfree(d_ptr, cs); dfree(d_changed, cs); dfree(d_done, cs);
        }
        cudaEventRecord(ev[3], cs);
        // compact the BlockRec array to stream order without gaps: rebase through a gather of summaries
        // (BlockRecs stay where they are; blk index -> record via descs[stream].blk_base + k)
        BlkSummary* d_summ = nullptr;
        BlockRec* d_compact = nullptr;
        D4_CUDA_CHECK(dalloc(&d_compact, nblk_total, cs));
        if (nblk_total) LAUNCH(k_compact_blocks, (unsigned)((nblk_total * 32 + 255) / 256), 256, cs, d_descs, d_blocks, d_jobs, nblk_total, d_compact);
        dfree(d_blocks, cs);
        d_blocks = d_compact;
        D4_CUDA_CHECK(dalloc(&d_summ, nblk_total, cs));
        summ.resize(nblk_total);
        if (nblk_total) LAUNCH(k_blk_summary, (unsigned)((nblk_total + 255) / 256), 256, cs, d_blocks, d_summ, nblk_total);
        D4_CUDA_CHECK(cudaMemcpyAsync(summ.data(), d_summ, sizeof(BlkSummary) * nblk_total, cudaMemcpyDeviceToHost, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(winfos.data(), d_infos, sizeof(StreamInfo) * W, cudaMemcpyDeviceToHost, cs));
        D4_CUDA_CHECK(cudaStreamSynchronize(cs));
        // k_emit flags a match that reaches before the start of its stream on the walker that saw it
        for (uint32_t i = 0; i < n; i++)
            for (uint32_t c = chain_off[i]; c < chain_off[i + 1]; c++)
                if (winfos[chain[c]].status != ST_OK && infos[i].status == ST_OK) infos[i].status = ST_PARSE;
        dfree(d_summ, cs); dfree(d_jobs, cs); dfree(d_chunks, cs);
        {
            const int rc = init_model(sblk_base);
            if (rc) return rc;
        }
        float t;
        cudaEventElapsedTime(&t, ev[0], ev[1]); ms[0] = t;
        cudaEventElapsedTime(&t, ev[1], ev[2]); ms[1] = t;
        cudaEventElapsedTime(&t, ev[2], ev[3]); ms[2] = t;
        ms[7] = (float)parse_rewalks;  // walkers whose guessed start was wrong or missing
        for (auto& e : ev) cudaEventDestroy(e);
        parsed = true;
        return DEFT4CU_OK;
    }

    // the optimiser's model of a batch whose blocks, symbols and decoded bytes are in place (parse() and compress()):
    // mask offsets, per-stream state and the BlkState of every block
    int init_model(const std::vector<uint64_t>& sblk_base) {
        mask_offs.resize(nblk_total);
        uint64_t mo = 0;
        for (uint64_t b = 0; b < nblk_total; b++) { mask_offs[b] = mo; mo += (summ[b].n_sym + 31) / 32; }
        maskwords_total = mo;
        sstate.assign(n, StreamState{});
        size_bits_in.assign(n, 0);
        for (uint32_t i = 0; i < n; i++) {
            StreamState& s = sstate[i];
            s.blk_base = sblk_base[i];
            s.status = infos[i].status;
            s.n_blocks = infos[i].status == ST_OK ? infos[i].n_blocks : 0;
            s.cut = s.n_blocks;
            s.total_bits = infos[i].total_bits;
            size_bits_in[i] = (int64_t)infos[i].total_bits;
        }
        uint64_t* d_moffs = nullptr;
        D4_CUDA_CHECK(dalloc(&d_moffs, nblk_total, cs));
        D4_CUDA_CHECK(dalloc(&d_blk_stream, nblk_total, cs));
        D4_CUDA_CHECK(dalloc(&d_bs, nblk_total, cs));
        D4_CUDA_CHECK(dalloc(&d_logs, nblk_total, cs));
        D4_CUDA_CHECK(dalloc(&d_maskpool, mo + 2, cs));
        D4_CUDA_CHECK(dalloc(&d_sstate, n, cs));
        D4_CUDA_CHECK(cudaMemsetAsync(d_maskpool, 0, (mo + 2) * 4, cs));
        // the stream states go to the device now as well: a handle may be written before it is optimised
        D4_CUDA_CHECK(cudaMemcpyAsync(d_sstate, sstate.data(), sizeof(StreamState) * n, cudaMemcpyHostToDevice, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(d_moffs, mask_offs.data(), 8 * nblk_total, cudaMemcpyHostToDevice, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(d_blk_stream, blk_stream.data(), 4 * nblk_total, cudaMemcpyHostToDevice, cs));
        if (nblk_total) LAUNCH(k_init_state, (unsigned)((nblk_total + 127) / 128), 128, cs, d_blocks, d_moffs, d_bs, nblk_total);
        D4_CUDA_CHECK(cudaStreamSynchronize(cs));
        dfree(d_moffs, cs);
        return DEFT4CU_OK;
    }

    // ---- compress: raw input bytes -> the model of their fixed-coded stream (lzrule.cuh, lzcomp.cuh) ----------------
    int compress(uint32_t bytes_per_block) {
        HostTimer ht("compress");
        release_model();
        too_big = false;
        block_bytes = bytes_per_block;
        cudaEvent_t ev[3];
        for (auto& e : ev) cudaEventCreate(&e);
        descs.assign(n + 1, StreamDesc{});
        infos.assign(n, StreamInfo{});
        D4_CUDA_CHECK(dalloc(&d_gerr, 8, cs));
        D4_CUDA_CHECK(cudaMemsetAsync(d_gerr, 0, 8 * sizeof(int), cs));
        // decoded bytes: the input itself, packed the way parse() packs them
        uint64_t ob = 0;
        for (uint32_t i = 0; i < n; i++) {
            descs[i].out_base = ob;
            infos[i].status = in_len[i] > 0xF0000000ull ? ST_UNSUPPORTED : ST_OK;
            if (infos[i].status == ST_OK) ob += in_len[i];
        }
        descs[n].out_base = ob;
        nout_total = ob;
        uint64_t ob_max = 0xF8000000ull;   // decoded offsets are 32-bit
        if (const char* e = getenv("D4_MAX_DECODED")) ob_max = std::min<uint64_t>(ob_max, strtoull(e, nullptr, 10));   // tests force the split
        if (ob >= ob_max) {
            too_big = true;
            for (uint32_t i = 0; i < n; i++) if (infos[i].status == ST_OK) infos[i].status = ST_UNSUPPORTED;
            set_error("decoded size of the batch exceeds 4 GiB; split the batch");
            return DEFT4CU_ERR_UNSUPPORTED;
        }
        D4_CUDA_CHECK(dalloc(&d_out, ob + 16, cs));
        for (uint32_t i = 0; i < n; i++)
            if (infos[i].status == ST_OK && in_len[i])
                D4_CUDA_CHECK(cudaMemcpyAsync(d_out + descs[i].out_base, d_in + in_off[i], in_len[i], cudaMemcpyDeviceToDevice, cs));
        // blocks of `bytes_per_block` input bytes, the last one shorter; an empty stream is one block holding only EOB
        std::vector<LzJob> jobs;
        std::vector<uint64_t> sblk_base(n);
        blk_stream.clear();
        for (uint32_t i = 0; i < n; i++) {
            sblk_base[i] = jobs.size();
            if (infos[i].status != ST_OK) continue;
            const uint64_t len = in_len[i], nb = len ? (len + bytes_per_block - 1) / bytes_per_block : 1;
            for (uint64_t k = 0; k < nb; k++) {
                LzJob jb{};
                jb.base = descs[i].out_base; jb.n = len;
                jb.s = (uint32_t)(k * bytes_per_block); jb.e = (uint32_t)std::min<uint64_t>(len, (k + 1) * bytes_per_block);
                jb.bfinal = k + 1 == nb;
                jobs.push_back(jb);
                blk_stream.push_back(i);
            }
        }
        nblk_total = jobs.size();
        LzJob* d_jobs = nullptr;
        LzRes* d_res = nullptr;
        uint32_t* d_m = nullptr;
        uint2* d_ent = nullptr;
        uint16_t* d_slab = nullptr;
        unsigned* d_counter = nullptr;
        D4_CUDA_CHECK(dalloc(&d_jobs, nblk_total, cs));
        D4_CUDA_CHECK(dalloc(&d_res, nblk_total, cs));
        D4_CUDA_CHECK(dalloc(&d_m, ob + 1, cs));
        D4_CUDA_CHECK(dalloc(&d_ent, nblk_total * LZ_NT, cs));
        D4_CUDA_CHECK(dalloc(&d_counter, 1, cs));
        D4_CUDA_CHECK(cudaMemsetAsync(d_counter, 0, 4, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(LzJob) * nblk_total, cudaMemcpyHostToDevice, cs));
        int perSM = 0;
        D4_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_lz_match, LZ_NT, LZ_SMEM));
        const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(nblk_total, (uint64_t)g_sms * std::max(perSM, 1)));
        D4_CUDA_CHECK(dalloc(&d_slab, (size_t)grid * LZ_WIN_CAP, cs));
        cudaEventRecord(ev[0], cs);
        if (nblk_total) LAUNCH_SM(k_lz_match, grid, LZ_NT, LZ_SMEM, cs, d_jobs, (uint32_t)nblk_total, d_out, d_m, d_slab, d_ent, d_res, d_counter);
        cudaEventRecord(ev[1], cs);
        std::vector<LzRes> lres(nblk_total);
        D4_CUDA_CHECK(cudaMemcpyAsync(lres.data(), d_res, sizeof(LzRes) * nblk_total, cudaMemcpyDeviceToHost, cs));
        D4_CUDA_CHECK(cudaStreamSynchronize(cs));
        if (stage && cs == own_cs) { host_release(stage); stage = nullptr; }   // upload()'s copy is behind us
        dfree(d_slab, cs); dfree(d_counter, cs);
        // symbol pool bases and block positions: exclusive scans over the batch and over each stream
        uint64_t sb = 0;
        summ.resize(nblk_total);
        for (uint32_t i = 0; i < n; i++) {
            descs[i].sym_base = sb;
            StreamInfo& si = infos[i];
            if (si.status != ST_OK) continue;
            uint64_t bit = 0;
            const uint64_t nb = (i + 1 < n ? sblk_base[i + 1] : nblk_total) - sblk_base[i];
            for (uint64_t k = sblk_base[i]; k < sblk_base[i] + nb; k++) {
                jobs[k].sym_base = sb; jobs[k].hdr_bit = bit;
                sb += lres[k].n_sym;
                bit += 3 + lres[k].payload;
                summ[k] = BlkSummary{1u, lres[k].n_sym, jobs[k].e - jobs[k].s, 1u, 0u};
                si.n_syms += lres[k].n_sym;
            }
            si.n_blocks = (uint32_t)nb;
            si.out_len = in_len[i];
            si.consumed = in_len[i];
            si.total_bits = si.end_bit = bit;
            si.final_seen = 1;
        }
        descs[n].sym_base = sb;
        nsym_total = sb;
        D4_CUDA_CHECK(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(LzJob) * nblk_total, cudaMemcpyHostToDevice, cs));
        D4_CUDA_CHECK(dalloc(&d_sym, sb, cs));
        D4_CUDA_CHECK(dalloc(&d_symout, sb, cs));
        D4_CUDA_CHECK(dalloc(&d_blocks, nblk_total, cs));
        if (nblk_total) LAUNCH(k_lz_emit, (unsigned)nblk_total, LZ_NT, cs, d_jobs, d_out, d_m, d_ent, d_res, d_sym, d_symout, d_blocks);
        cudaEventRecord(ev[2], cs);
        dfree(d_jobs, cs); dfree(d_res, cs); dfree(d_m, cs); dfree(d_ent, cs);
        {
            const int rc = init_model(sblk_base);
            if (rc) return rc;
        }
        float t;
        cudaEventElapsedTime(&t, ev[0], ev[1]); ms[0] = t;   // match + parse
        cudaEventElapsedTime(&t, ev[1], ev[2]); ms[1] = t;   // emit (and the host scan between them)
        ms[2] = 0; ms[7] = 0;
        for (auto& e : ev) cudaEventDestroy(e);
        parsed = true;
        compressed = true;
        return DEFT4CU_OK;
    }

    // per-CTA engine scratch: one contiguous, 2 MiB aligned slab per CTA (engine.cuh eng_scratch_layout)
    // Every CTA gets a slab sized for the largest job, so one large stream among many small ones would ask for grid times
    // its slab.  The kernels take their jobs from a counter, so `grid` is lowered to what the device can hold (free
    // memory plus what the stream-ordered pool keeps in reserve, less a margin); fewer CTAs only take longer.
    unsigned char* scratch_raw = nullptr;
    cudaError_t alloc_scratch(EngScratch& sc, unsigned& grid, uint32_t maxwords, uint64_t maxu) {
        const size_t stride = eng_scratch_layout(sc, maxwords, maxu);
        const size_t align = (size_t)2 << 20;
        size_t freeb = 0, totalb = 0;
        if (cudaMemGetInfo(&freeb, &totalb) == cudaSuccess) {
            cudaMemPool_t pool;
            uint64_t res = 0, used = 0;
            if (cudaDeviceGetDefaultMemPool(&pool, g_device) == cudaSuccess &&
                cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &res) == cudaSuccess &&
                cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && res > used)
                freeb += (size_t)(res - used);
            const size_t margin = ((size_t)1 << 30) + totalb / 16;
            const size_t fit = freeb > margin + align ? (freeb - margin - align) / stride : 0;
            grid = (unsigned)std::max<size_t>(1, std::min<size_t>(grid, fit));
        }
        cudaError_t e = dalloc(&scratch_raw, stride * grid + align, cs);
        if (e != cudaSuccess) return e;
        sc.slab = (unsigned char*)(((uintptr_t)scratch_raw + align - 1) & ~(uintptr_t)(align - 1));
        if (getenv("D4_POISON")) cudaMemsetAsync(sc.slab, 0x7F, stride * grid, cs);
        return cudaSuccess;
    }
    void free_scratch(EngScratch&) { dfree(scratch_raw, cs); }

    // ---- optimise: phase A over blocks, then per-stream replay/merge/layout ----------------------------
    int optimise(uint32_t flags, const std::vector<uint8_t>& selected) {
        HostTimer ht("optimise");
        cudaEvent_t ev[3];
        for (auto& e : ev) cudaEventCreate(&e);
        const int merge = (flags & DEFT4CU_MERGE_BLOCKS) ? 1 : 0;
        if (optimised && nblk_total) {
            // DeflateStream.optimise may be called again on the same object (DeflateStream.java:496): the block list is
            // the current model's (merged, removed and stored blocks), not the parsed one
            BlkSummary* d_summ = nullptr;
            D4_CUDA_CHECK(dalloc(&d_summ, nblk_total, cs));
            LAUNCH(k_state_summary, (unsigned)((nblk_total + 255) / 256), 256, cs, d_bs, d_summ, nblk_total);
            D4_CUDA_CHECK(cudaMemcpyAsync(summ.data(), d_summ, sizeof(BlkSummary) * nblk_total, cudaMemcpyDeviceToHost, cs));
            D4_CUDA_CHECK(cudaStreamSynchronize(cs));
            dfree(d_summ, cs);
        }
        optimised = true;
        std::vector<uint32_t> jobs;
        uint32_t maxsym = 1, maxstream = 1;
        uint64_t maxout = 1, maxstream_out = 1;
        for (uint32_t i = 0; i < n; i++) {
            StreamState& s = sstate[i];
            s.selected = selected[i] && s.status == ST_OK;
            s.saved_bits = 0;
            if (!s.selected) continue;
            uint64_t ssum = 0;
            // blocks [0, cut) take part in phase A: the loop of DeflateStream.optimise ends at the first empty block it
            // removes (SURVEY.md H6); a sole block is optimised even when empty (:510)
            uint32_t n_alive = 0;
            for (uint32_t k = 0; k < s.n_blocks; k++) n_alive += summ[s.blk_base + k].alive;
            s.cut = s.n_blocks;
            for (uint32_t k = 0; k < s.n_blocks; k++) {
                const BlkSummary& b = summ[s.blk_base + k];
                if (b.alive && b.out_len == 0 && n_alive != 1) { s.cut = k; break; }
            }
            for (uint32_t k = 0; k < s.n_blocks; k++) {
                const BlkSummary& b = summ[s.blk_base + k];
                ssum += b.n_sym;
                if (k < s.cut && b.type != 0 && b.alive) {
                    jobs.push_back((uint32_t)(s.blk_base + k));
                    maxsym = std::max(maxsym, b.n_sym);
                    maxout = std::max<uint64_t>(maxout, b.out_len);
                }
            }
            maxstream = (uint32_t)std::max<uint64_t>(maxstream, ssum);
            maxstream_out = std::max<uint64_t>(maxstream_out, infos[i].out_len);
        }
        const bool tracing = g_trace_dev != nullptr;
        if (!tracing) std::stable_sort(jobs.begin(), jobs.end(), [&](uint32_t a, uint32_t b) { return summ[a].n_sym > summ[b].n_sym; });
        D4_CUDA_CHECK(cudaMemcpyAsync(d_sstate, sstate.data(), sizeof(StreamState) * n, cudaMemcpyHostToDevice, cs));
        cudaEventRecord(ev[0], cs);
        if (!jobs.empty()) {
            uint32_t* d_jobs = nullptr;
            unsigned* d_counter = nullptr;
            D4_CUDA_CHECK(dalloc(&d_jobs, jobs.size(), cs));
            D4_CUDA_CHECK(dalloc(&d_counter, 1, cs));
            D4_CUDA_CHECK(cudaMemsetAsync(d_counter, 0, 4, cs));
            D4_CUDA_CHECK(cudaMemcpyAsync(d_jobs, jobs.data(), 4 * jobs.size(), cudaMemcpyHostToDevice, cs));
            int perSM = 0;
            cudaFuncSetAttribute(k_opt_blocks, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            D4_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_opt_blocks, ENG_NT, 0));
            if (perSM < 1) perSM = 1;
            if (const char* e = getenv("D4_CTAS_PER_SM")) perSM = std::max(1, std::min(perSM, atoi(e)));  // A/B knob
            unsigned grid = (unsigned)std::min<uint64_t>(jobs.size(), (uint64_t)g_sms * perSM);
            if (tracing) grid = 1;
            EngScratch sc{};
            D4_CUDA_CHECK(alloc_scratch(sc, grid, (maxsym + 31) / 32 + 1, maxout));
            g_opt_launches++;
            LAUNCH(k_opt_blocks, grid, ENG_NT, cs, d_jobs, (uint32_t)jobs.size(), d_bs, d_logs, d_sym, d_symout, d_out, d_maskpool, sc, d_counter, d_gerr);
            free_scratch(sc);
            dfree(d_jobs, cs); dfree(d_counter, cs);
        }
        cudaEventRecord(ev[1], cs);
        {
            EngScratch sc{};
            int perSM = 0;
            cudaFuncSetAttribute(k_finish, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            D4_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_finish, ENG_NT, 0));
            if (perSM < 1) perSM = 1;
            unsigned grid = (unsigned)std::min<uint64_t>(n, (uint64_t)g_sms * perSM);
            unsigned* d_counter = nullptr;
            D4_CUDA_CHECK(dalloc(&d_counter, 1, cs));
            D4_CUDA_CHECK(cudaMemsetAsync(d_counter, 0, 4, cs));
            if (merge) D4_CUDA_CHECK(alloc_scratch(sc, grid, (maxstream + 31) / 32 + 2, maxstream_out));
            if (n) LAUNCH(k_finish, grid, ENG_NT, cs, d_sstate, n, d_bs, d_logs, d_sym, d_symout, d_out, d_maskpool, sc, merge, d_counter, d_gerr);
            if (merge) free_scratch(sc);
            dfree(d_counter, cs);
        }
        cudaEventRecord(ev[2], cs);
        int gerrv[8] = {0};
        D4_CUDA_CHECK(cudaMemcpyAsync(sstate.data(), d_sstate, sizeof(StreamState) * n, cudaMemcpyDeviceToHost, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(gerrv, d_gerr, sizeof(gerrv), cudaMemcpyDeviceToHost, cs));
        D4_CUDA_CHECK(cudaStreamSynchronize(cs));
        float t;
        cudaEventElapsedTime(&t, ev[0], ev[1]); ms[3] = t;
        cudaEventElapsedTime(&t, ev[1], ev[2]); ms[4] = t;
        for (auto& e : ev) cudaEventDestroy(e);
        const int gerr = gerrv[0];
        if (gerr == 13 || gerr == 14) {
            char msg[256];
            snprintf(msg, sizeof msg, "engine self-check: block %d round %d winner idx %d selected size %d, materialised size %d (check %d: 1 "
                     "incumbent != previous winner, 2 payload, 3 size; previous %d; %zu jobs)",
                     gerrv[1], gerrv[2], gerrv[3], gerrv[4], gerrv[5], gerrv[6], gerrv[7], jobs.size());
            set_error(msg);
            return DEFT4CU_ERR_CUDA;
        }
        if (gerr) {
            set_error(gerr == ERR_ROUNDS ? "optimiser hit an internal limit: more than 64 optimiseBlock rounds on one block"
                      : gerr == ERR_POOL ? "optimiser: internal table pool overflow"
                      : gerr == ERR_INTERNAL ? "optimiser: enumerator/executor protocol error (internal)"
                                         : "optimiser: a Huffman tree could not be balanced (the reference throws here)");
            D4_CUDA_CHECK(cudaMemsetAsync(d_gerr, 0, sizeof(int), cs));
            for (uint32_t i = 0; i < n; i++) if (sstate[i].selected) sstate[i].status = ST_UNSUPPORTED;
            return DEFT4CU_ERR_UNSUPPORTED;
        }
        dfree(d_dst, cs);  // stale output
        h_dst.clear();
        return DEFT4CU_OK;
    }

    // ---- write ---------------------------------------------------------------------------------------
    int write() {
        HostTimer ht("write");
        cudaEvent_t ev[2];
        for (auto& e : ev) cudaEventCreate(&e);
        dst_off.assign(n, 0); dst_len.assign(n, 0);
        uint64_t off = 0;
        for (uint32_t i = 0; i < n; i++) {
            dst_off[i] = off;
            if (sstate[i].status != ST_OK) continue;
            dst_len[i] = (sstate[i].total_bits + 7) / 8;
            off += (dst_len[i] + 16 + 7) & ~7ull;
        }
        dst_total = off + 8;
        dfree(d_dst, cs); dfree(d_dst_off, cs);
        h_dst.clear();
        D4_CUDA_CHECK(dalloc(&d_dst, dst_total, cs));
        D4_CUDA_CHECK(dalloc(&d_dst_off, n, cs));
        D4_CUDA_CHECK(cudaMemsetAsync(d_dst, 0, dst_total, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(d_dst_off, dst_off.data(), 8 * n, cudaMemcpyHostToDevice, cs));
        cudaEventRecord(ev[0], cs);
        if (nblk_total)
            LAUNCH(k_write, (unsigned)nblk_total, WR_NT, cs, d_sstate, d_blk_stream, d_bs, d_sym, d_symout, d_out, d_maskpool, d_dst_off,
                   (unsigned long long*)d_dst, d_gerr);
        cudaEventRecord(ev[1], cs);
        int gerr[8] = {0};
        D4_CUDA_CHECK(cudaMemcpyAsync(gerr, d_gerr, sizeof(gerr), cudaMemcpyDeviceToHost, cs));
        D4_CUDA_CHECK(cudaStreamSynchronize(cs));
        float t;
        cudaEventElapsedTime(&t, ev[0], ev[1]); ms[5] = t;
        for (auto& e : ev) cudaEventDestroy(e);
        if (gerr[0]) {
            char msg[200];
            snprintf(msg, sizeof msg, "writer and cost model disagree (code %d) on block %d: wrote %d bits, model says %d (%s)",
                     gerr[0], gerr[1], gerr[2], gerr[3], gerr[4] == 1 ? "header" : "block");
            set_error(msg);
            return DEFT4CU_ERR_WRITE;
        }
        return DEFT4CU_OK;
    }

    int checksums() {
        if (have_sums) return DEFT4CU_OK;
        HostTimer ht("checksums");
        static std::once_flag once;
        std::call_once(once, [] { k_crc_init<<<1, 1>>>(); cudaDeviceSynchronize(); });
        cudaEvent_t ev[2];
        for (auto& e : ev) cudaEventCreate(&e);
        std::vector<uint64_t> off(n), len(n);
        std::vector<CkJob> jobs;
        for (uint32_t i = 0; i < n; i++) {
            off[i] = descs[i].out_base; len[i] = infos[i].status == ST_OK ? infos[i].out_len : 0;
            const uint64_t c0 = off[i] >> CK_CELL_LOG2, c1 = (off[i] + len[i]) >> CK_CELL_LOG2;
            const uint64_t cells = c1 > c0 ? c1 - c0 : 0;
            const uint32_t nj = (uint32_t)std::max<uint64_t>(1, (cells + CK_NT - 1) / CK_NT);
            for (uint32_t c = 0; c < nj; c++) jobs.push_back(CkJob{i, c});
        }
        uint64_t *d_off = nullptr, *d_len = nullptr;
        uint32_t *d_crc = nullptr, *d_ad = nullptr;
        CkJob* d_jobs = nullptr;
        CkAcc* d_acc = nullptr;
        D4_CUDA_CHECK(dalloc(&d_off, n, cs)); D4_CUDA_CHECK(dalloc(&d_len, n, cs));
        D4_CUDA_CHECK(dalloc(&d_crc, n, cs)); D4_CUDA_CHECK(dalloc(&d_ad, n, cs));
        D4_CUDA_CHECK(dalloc(&d_jobs, jobs.size(), cs)); D4_CUDA_CHECK(dalloc(&d_acc, n, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(d_off, off.data(), 8 * n, cudaMemcpyHostToDevice, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(d_len, len.data(), 8 * n, cudaMemcpyHostToDevice, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(CkJob) * jobs.size(), cudaMemcpyHostToDevice, cs));
        D4_CUDA_CHECK(cudaMemsetAsync(d_acc, 0, sizeof(CkAcc) * std::max<uint32_t>(n, 1), cs));
        cudaEventRecord(ev[0], cs);
        if (n) {
            LAUNCH(k_checksum_cells, (unsigned)jobs.size(), CK_NT, cs, d_out, d_off, d_len, d_jobs, d_acc);
            LAUNCH(k_checksum_final, (n * 32 + 255) / 256, 256, cs, d_len, d_acc, n, d_crc, d_ad);
        }
        cudaEventRecord(ev[1], cs);
        crc.resize(n); adler.resize(n);
        D4_CUDA_CHECK(cudaMemcpyAsync(crc.data(), d_crc, 4 * n, cudaMemcpyDeviceToHost, cs));
        D4_CUDA_CHECK(cudaMemcpyAsync(adler.data(), d_ad, 4 * n, cudaMemcpyDeviceToHost, cs));
        D4_CUDA_CHECK(cudaStreamSynchronize(cs));
        float t;
        cudaEventElapsedTime(&t, ev[0], ev[1]); ms[6] = t;
        for (auto& e : ev) cudaEventDestroy(e);
        dfree(d_off, cs); dfree(d_len, cs); dfree(d_crc, cs); dfree(d_ad, cs); dfree(d_jobs, cs); dfree(d_acc, cs);
        have_sums = true;
        return DEFT4CU_OK;
    }
};

}  // namespace d4

using namespace d4;

struct deft4cu_stream {
    std::shared_ptr<Batch> batch;
    uint32_t idx;
    bool written = false;
};
struct deft4cu_device_batch {
    std::shared_ptr<Batch> batch;
};

extern "C" {

int deft4cu_init(int device) {
    std::lock_guard<std::mutex> lk(g_mu);
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error(std::string("no CUDA device: ") + cudaGetErrorString(e));
        return DEFT4CU_ERR_CUDA;
    }
    if (device < 0 || device >= count) { set_error("bad device index"); return DEFT4CU_ERR_ARG; }
    D4_CUDA_CHECK(cudaSetDevice(device));
    cudaDeviceProp p;
    D4_CUDA_CHECK(cudaGetDeviceProperties(&p, device));
    g_sms = p.multiProcessorCount;
    D4_CUDA_CHECK(cudaFuncSetAttribute(k_count, cudaFuncAttributeMaxDynamicSharedMemorySize, WIN_BYTES + WIN_SLACK + 16));
    D4_CUDA_CHECK(cudaFuncSetAttribute(k_lz_match, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM));
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    if (getenv("D4_DEBUG_LIMITS")) {
        size_t st = 0, hp = 0;
        cudaDeviceGetLimit(&st, cudaLimitStackSize);
        cudaDeviceGetLimit(&hp, cudaLimitMallocHeapSize);
        cudaFuncAttributes fa;
        cudaFuncGetAttributes(&fa, k_opt_blocks);
        fprintf(stderr, "[deft4cu] stack limit %zu heap %zu; k_opt_blocks local %zu regs %d smem %zu\n", st, hp, fa.localSizeBytes, fa.numRegs, fa.sharedSizeBytes);
        if (getenv("D4_STACK")) { cudaDeviceSetLimit(cudaLimitStackSize, atoi(getenv("D4_STACK"))); }
    }
    g_device = device;
    return DEFT4CU_OK;
}
const char* deft4cu_last_error(void) { return g_err.c_str(); }
const char* deft4cu_version(void) { return "deft4cu 0.2 (sm_100a)"; }

// ---- parity-debug trace (engine.cuh g_trace) ---------------------------------------------------------------
int deft4cu_debug_trace_begin(uint32_t cap) {
    int rc = ensure_init();
    if (rc) return rc;
    if (g_trace_dev) { cudaFree(g_trace_dev); g_trace_dev = nullptr; }
    D4_CUDA_CHECK(cudaMalloc((void**)&g_trace_dev, 16ull * cap));
    g_trace_dev_cap = cap;
    unsigned zero = 0;
    D4_CUDA_CHECK(cudaMemcpyToSymbol(g_trace, &g_trace_dev, sizeof(g_trace_dev)));
    D4_CUDA_CHECK(cudaMemcpyToSymbol(g_trace_cap, &cap, sizeof(cap)));
    D4_CUDA_CHECK(cudaMemcpyToSymbol(g_trace_n, &zero, sizeof(zero)));
    return DEFT4CU_OK;
}
int deft4cu_debug_trace_end(int64_t* dst, uint32_t cap, uint32_t* n) {
    if (!g_trace_dev) { set_error("trace not armed"); return DEFT4CU_ERR_ARG; }
    D4_CUDA_CHECK(cudaDeviceSynchronize());
    unsigned cnt = 0;
    D4_CUDA_CHECK(cudaMemcpyFromSymbol(&cnt, g_trace_n, sizeof(cnt)));
    long long* null = nullptr;
    D4_CUDA_CHECK(cudaMemcpyToSymbol(g_trace, &null, sizeof(null)));
    if (n) *n = cnt;
    uint32_t m = std::min(std::min(cnt, cap), g_trace_dev_cap);
    if (m) D4_CUDA_CHECK(cudaMemcpy(dst, g_trace_dev, 16ull * m, cudaMemcpyDeviceToHost));
    cudaFree(g_trace_dev);
    g_trace_dev = nullptr;
    return DEFT4CU_OK;
}

// how many times the candidate engine kernel has been launched (a list of streams should cost ONE launch)
uint64_t deft4cu_debug_engine_launches(void) { return g_opt_launches; }

// cycle counters of a -DD4_PROF build (engine.cuh g_prof); returns DEFT4CU_ERR_ARG in ordinary builds
int deft4cu_debug_prof(uint64_t* dst, uint32_t n, int reset) {
#ifdef D4_PROF
    unsigned long long h[64];
    D4_CUDA_CHECK(cudaDeviceSynchronize());
    D4_CUDA_CHECK(cudaMemcpyFromSymbol(h, g_prof, sizeof(h)));
    for (uint32_t i = 0; i < n && i < 64; i++) dst[i] = h[i];
    if (reset) { memset(h, 0, sizeof h); D4_CUDA_CHECK(cudaMemcpyToSymbol(g_prof, h, sizeof(h))); }
    return DEFT4CU_OK;
#else
    (void)dst; (void)n; (void)reset;
    set_error("not a -DD4_PROF build");
    return DEFT4CU_ERR_ARG;
#endif
}

// ---- handle API ------------------------------------------------------------------------------------------
int deft4cu_stream_parse_batch(const uint8_t* const* data, const uint64_t* len, uint32_t n, deft4cu_stream** handles,
                               int32_t* status, uint64_t* consumed) {
    int rc = ensure_init();
    if (rc) return rc;
    auto b = std::make_shared<Batch>();
    rc = b->upload(data, len, n);
    if (rc) return rc;
    rc = b->parse();
    if (rc && rc != DEFT4CU_ERR_UNSUPPORTED) return rc;
    for (uint32_t i = 0; i < n; i++) {
        int st = b->infos[i].status;
        if (status) status[i] = st;
        if (consumed) consumed[i] = b->infos[i].consumed;
        handles[i] = nullptr;
        if (st == ST_OK) handles[i] = new deft4cu_stream{b, i};
    }
    return DEFT4CU_OK;
}
static int compress_block_bytes(uint32_t* block_bytes) {
    if (*block_bytes == 0) *block_bytes = LZ_BLOCK_DEFAULT;
    if (*block_bytes < LZ_BLOCK_MIN || *block_bytes > LZ_BLOCK_MAX) {
        set_error("block_bytes must be 0 (default) or within [256, 65535]");
        return DEFT4CU_ERR_ARG;
    }
    return DEFT4CU_OK;
}
int deft4cu_stream_compress_batch(const uint8_t* const* data, const uint64_t* len, uint32_t n, uint32_t block_bytes,
                                  deft4cu_stream** handles, int32_t* status) {
    int rc = compress_block_bytes(&block_bytes);
    if (rc) return rc;
    rc = ensure_init();
    if (rc) return rc;
    auto b = std::make_shared<Batch>();
    rc = b->upload(data, len, n);
    if (rc) return rc;
    rc = b->compress(block_bytes);
    if (rc && rc != DEFT4CU_ERR_UNSUPPORTED) return rc;
    for (uint32_t i = 0; i < n; i++) {
        const int st = b->infos[i].status;
        if (status) status[i] = st;
        handles[i] = nullptr;
        if (st == ST_OK) handles[i] = new deft4cu_stream{b, i};
    }
    return DEFT4CU_OK;
}
int deft4cu_stream_parse(const uint8_t* data, uint64_t len, deft4cu_stream** out, uint64_t* consumed) {
    int32_t st = 0;
    uint64_t c = 0;
    *out = nullptr;
    int rc = deft4cu_stream_parse_batch(&data, &len, 1, out, &st, &c);
    if (consumed) *consumed = c;
    if (rc) return rc;
    return st;
}
void deft4cu_stream_free(deft4cu_stream* s) { delete s; }

int deft4cu_stream_optimise_batch(deft4cu_stream* const* s, uint32_t n, uint32_t flags, int64_t* saved_bits) {
    // group by batch
    std::vector<Batch*> batches;
    for (uint32_t i = 0; i < n; i++) {
        if (!s[i]) return DEFT4CU_ERR_ARG;
        if (std::find(batches.begin(), batches.end(), s[i]->batch.get()) == batches.end()) batches.push_back(s[i]->batch.get());
    }
    // The reference's batch point is the stream LIST (DeflateFilesContainer.optimise, DeflateFilesContainer.java:18-43),
    // but containers parse their streams one at a time (each parse must report where the stream ended), so the list
    // usually arrives as one batch per stream.  Streams that have not been optimised yet are regrouped into ONE batch
    // (device-to-device copy of their input, parsed again together): one launch of every kernel for the whole list.
    if (batches.size() > 1) {
        // A compressed batch's input is raw data: batches are regrouped only when all of them were parsed, or all of them
        // were compressed with the same block size (and then compressed again together)
        bool fresh = true;
        for (Batch* b : batches)
            fresh = fresh && !b->optimised && b->parsed && b->compressed == batches[0]->compressed &&
                    b->block_bytes == batches[0]->block_bytes;
        for (uint32_t i = 0; i < n && fresh; i++)
            for (uint32_t k = 0; k < i; k++) if (s[k] == s[i]) fresh = false;   // a handle listed twice
        if (fresh) {
            std::vector<std::pair<Batch*, uint32_t>> src(n);
            for (uint32_t i = 0; i < n; i++) src[i] = {s[i]->batch.get(), s[i]->idx};
            auto nb = std::make_shared<Batch>();
            int rc = nb->upload_from(src);
            if (rc == DEFT4CU_OK) rc = batches[0]->compressed ? nb->compress(batches[0]->block_bytes) : nb->parse();
            bool same = rc == DEFT4CU_OK;
            for (uint32_t i = 0; i < n && same; i++) same = nb->infos[i].status == ST_OK;
            if (same) {
                for (uint32_t i = 0; i < n; i++) { s[i]->batch = nb; s[i]->idx = i; }
                batches.assign(1, nb.get());
            } else if (rc != DEFT4CU_OK && rc != DEFT4CU_ERR_UNSUPPORTED) return rc;
            // (too large for one batch, or a stream that no longer parses: keep the batches as they are)
        }
    }
    int worst = DEFT4CU_OK;
    for (Batch* b : batches) {
        std::vector<uint8_t> sel(b->n, 0);
        for (uint32_t i = 0; i < n; i++) if (s[i]->batch.get() == b) sel[s[i]->idx] = 1;
        int rc = b->optimise(flags, sel);
        if (rc) worst = rc;
    }
    for (uint32_t i = 0; i < n; i++) {
        s[i]->written = false;
        if (saved_bits) saved_bits[i] = s[i]->batch->sstate[s[i]->idx].saved_bits;
    }
    return worst;
}
int deft4cu_stream_optimise(deft4cu_stream* s, uint32_t flags, int64_t* saved_bits) {
    return deft4cu_stream_optimise_batch(&s, 1, flags, saved_bits);
}
int64_t deft4cu_stream_size_bits(const deft4cu_stream* s) { return (int64_t)s->batch->sstate[s->idx].total_bits; }
uint64_t deft4cu_stream_uncompressed_len(const deft4cu_stream* s) { return s->batch->infos[s->idx].out_len; }
int deft4cu_stream_uncompressed(const deft4cu_stream* s, uint8_t* dst, uint64_t cap) {
    Batch& b = *s->batch;
    uint64_t len = b.infos[s->idx].out_len;
    if (cap < len) return DEFT4CU_ERR_ARG;
    if (len) D4_CUDA_CHECK(cudaMemcpyAsync(dst, b.d_out + b.descs[s->idx].out_base, len, cudaMemcpyDeviceToHost, b.cs));
    D4_CUDA_CHECK(cudaStreamSynchronize(b.cs));
    return DEFT4CU_OK;
}
int deft4cu_stream_checksums(const deft4cu_stream* s, uint32_t* crc32, uint32_t* adler32) {
    Batch& b = *s->batch;
    int rc = b.checksums();
    if (rc) return rc;
    if (crc32) *crc32 = b.crc[s->idx];
    if (adler32) *adler32 = b.adler[s->idx];
    return DEFT4CU_OK;
}
int deft4cu_stream_write(const deft4cu_stream* s, uint8_t* dst, uint64_t cap, uint64_t* len) {
    Batch& b = *s->batch;
    if (b.sstate[s->idx].status != ST_OK) return DEFT4CU_ERR_WRITE;
    if (!b.d_dst) {
        int rc = b.write();
        if (rc) return rc;
    }
    uint64_t l = b.dst_len[s->idx];
    if (len) *len = l;
    if (dst && cap >= l) {
        // a container asks stream by stream (PNGFile/ZipFile.write): the whole batch comes over in one copy the first time
        if (b.n > 1 && b.dst_total <= (1ull << 30)) {
            if (b.h_dst.empty()) {
                b.h_dst.resize(b.dst_total);
                D4_CUDA_CHECK(cudaMemcpyAsync(b.h_dst.data(), b.d_dst, b.dst_total, cudaMemcpyDeviceToHost, b.cs));
                D4_CUDA_CHECK(cudaStreamSynchronize(b.cs));
            }
            if (l) memcpy(dst, b.h_dst.data() + b.dst_off[s->idx], l);
            return DEFT4CU_OK;
        }
        if (l) D4_CUDA_CHECK(cudaMemcpyAsync(dst, b.d_dst + b.dst_off[s->idx], l, cudaMemcpyDeviceToHost, b.cs));
        D4_CUDA_CHECK(cudaStreamSynchronize(b.cs));
    }
    return DEFT4CU_OK;
}

uint32_t deft4cu_stream_block_count(const deft4cu_stream* s) {
    Batch& b = *s->batch;
    const StreamState& st = b.sstate[s->idx];
    std::vector<BlkState> bs(st.n_blocks);
    if (st.n_blocks) cudaMemcpy(bs.data(), b.d_bs + st.blk_base, sizeof(BlkState) * st.n_blocks, cudaMemcpyDeviceToHost);
    uint32_t c = 0;
    for (auto& x : bs) c += x.alive ? 1 : 0;
    return c;
}
static int fetch_block(const deft4cu_stream* s, uint32_t block, BlkState* out) {
    Batch& b = *s->batch;
    const StreamState& st = b.sstate[s->idx];
    std::vector<BlkState> bs(st.n_blocks);
    if (st.n_blocks) cudaMemcpy(bs.data(), b.d_bs + st.blk_base, sizeof(BlkState) * st.n_blocks, cudaMemcpyDeviceToHost);
    uint32_t c = 0;
    for (auto& x : bs) {
        if (!x.alive) continue;
        if (c == block) { *out = x; return 0; }
        c++;
    }
    return 1;
}
// final symbol list of a block on the host (inspection only): expands replaced matches into literals
static int fetch_symbols(const deft4cu_stream* s, const BlkState& x, std::vector<int32_t>& triples) {
    Batch& b = *s->batch;
    std::vector<uint32_t> sym(x.n_sym), so(x.n_sym), mask((x.n_sym + 31) / 32 + 1);
    std::vector<uint8_t> out(x.out_len + 1);
    if (x.n_sym) {
        cudaMemcpy(sym.data(), b.d_sym + x.sym_off, 4ull * x.n_sym, cudaMemcpyDeviceToHost);
        cudaMemcpy(so.data(), b.d_symout + x.sym_off, 4ull * x.n_sym, cudaMemcpyDeviceToHost);
        cudaMemcpy(mask.data(), b.d_maskpool + x.mask_off, 4ull * ((x.n_sym + 31) / 32), cudaMemcpyDeviceToHost);
    }
    if (x.out_len) cudaMemcpy(out.data(), b.d_out + x.out_off, x.out_len, cudaMemcpyDeviceToHost);
    for (uint32_t i = 0; i < x.n_sym; i++) {
        uint32_t v = sym[i];
        if (!sym_is_match(v)) {
            if (v <= 256) { triples.push_back(0); triples.push_back((int32_t)v); triples.push_back(0); }
        } else if ((mask[i >> 5] >> (i & 31)) & 1) {
            for (int k = 0; k < sym_len(v); k++) {
                triples.push_back(0); triples.push_back(out[so[i] - x.out_off + k]); triples.push_back(0);
            }
        } else {
            triples.push_back(sym_dist(v)); triples.push_back(sym_len(v)); triples.push_back(sym_edge(v));
        }
    }
    return 0;
}
int deft4cu_stream_block_info(const deft4cu_stream* s, uint32_t block, deft4cu_block_info* o) {
    BlkState x;
    if (fetch_block(s, block, &x)) return DEFT4CU_ERR_ARG;
    memset(o, 0, sizeof *o);
    o->type = x.cand.tab.type;
    o->size_bits = x.size_bits;
    o->position = (int64_t)x.bit_pos;
    o->uncompressed_len = x.out_len;
    if (x.cand.tab.type != 0) {
        std::vector<int32_t> t;
        fetch_symbols(s, x, t);
        o->n_symbols = (uint32_t)(t.size() / 3);
        o->litlen_size_bits = x.cand.payload;
        if (x.cand.tab.type == 2) {
            o->n_rle_pairs = x.cand.hdr.np;
            o->num_litlen_lens = x.cand.tab.nL; o->num_dist_lens = x.cand.tab.nD; o->num_codelen_lens = x.cand.hdr.ncl;
            o->header_size_bits = x.cand.hdr.bits;
        }
    }
    return DEFT4CU_OK;
}
uint32_t deft4cu_stream_block_symbols(const deft4cu_stream* s, uint32_t block, int32_t* dst, uint32_t cap) {
    BlkState x;
    if (fetch_block(s, block, &x) || x.cand.tab.type == 0) return 0;
    std::vector<int32_t> t;
    fetch_symbols(s, x, t);
    uint32_t nsy = (uint32_t)(t.size() / 3);
    for (uint32_t i = 0; i < nsy && i < cap; i++) { dst[3 * i] = t[3 * i]; dst[3 * i + 1] = t[3 * i + 1]; dst[3 * i + 2] = t[3 * i + 2]; }
    return nsy;
}
uint32_t deft4cu_stream_block_rle_pairs(const deft4cu_stream* s, uint32_t block, int32_t* dst, uint32_t cap) {
    BlkState x;
    if (fetch_block(s, block, &x) || x.cand.tab.type != 2) return 0;
    for (uint32_t i = 0; i < x.cand.hdr.np && i < cap; i++) { dst[2 * i] = pair_run(x.cand.hdr.pairs[i]); dst[2 * i + 1] = pair_sym(x.cand.hdr.pairs[i]); }
    return x.cand.hdr.np;
}
uint32_t deft4cu_stream_block_codelens(const deft4cu_stream* s, uint32_t block, int which, int32_t* dst, uint32_t cap) {
    BlkState x;
    if (fetch_block(s, block, &x) || x.cand.tab.type == 0) return 0;
    uint32_t nn = which == 0 ? x.cand.tab.nL : which == 1 ? x.cand.tab.nD : (x.cand.tab.type == 2 ? 19 : 0);
    for (uint32_t i = 0; i < nn && i < cap; i++) dst[i] = which == 0 ? x.cand.tab.L[i] : which == 1 ? x.cand.tab.D[i] : x.cand.hdr.CL[i];
    return nn;
}

// ---- batch entry -------------------------------------------------------------------------------------------
static int fill_results(Batch& b, deft4cu_result* results, bool fetch_out) {
    int nout = 0;
    for (uint32_t i = 0; i < b.n; i++) {
        deft4cu_result& r = results[i];
        memset(&r, 0, sizeof r);
        r.status = b.sstate[i].status;
        r.consumed_bytes = b.infos[i].consumed;
        if (r.status != ST_OK) continue;
        r.saved_bits = b.sstate[i].saved_bits;
        r.uncompressed_len = b.infos[i].out_len;
        r.size_bits_in = b.size_bits_in[i];
        r.size_bits_out = (int64_t)b.sstate[i].total_bits;
        r.crc32 = b.crc.size() > i ? b.crc[i] : 0;
        r.adler32 = b.adler.size() > i ? b.adler[i] : 0;
        r.out_len = b.dst_len[i];
        nout++;
    }
    if (fetch_out && nout) {
        // the rewritten streams sit back to back in d_dst: one copy into one pinned block, `out` pointers into it
        uint8_t* blk = host_block_acquire(b.dst_total, nout);
        if (!blk) { set_error("out of host memory for the result buffers"); return DEFT4CU_ERR_CUDA; }
        D4_CUDA_CHECK(cudaMemcpyAsync(blk, b.d_dst, b.dst_total, cudaMemcpyDeviceToHost, b.cs));
        for (uint32_t i = 0; i < b.n; i++)
            if (results[i].status == ST_OK) results[i].out = blk + b.dst_off[i];
    }
    D4_CUDA_CHECK(cudaStreamSynchronize(b.cs));
    return DEFT4CU_OK;
}

int deft4cu_optimise_batch(const uint8_t* const* in, const uint64_t* in_len, uint32_t n, uint32_t flags, deft4cu_result* results) {
    int rc = ensure_init();
    if (rc) return rc;
    Batch b;
    rc = b.upload(in, in_len, n);
    if (rc) return rc;
    rc = b.parse();
    if (rc == DEFT4CU_ERR_UNSUPPORTED && b.too_big && n > 1) {
        // more than 4 GiB of decoded data: the list is optimised in two halves (streams never interact)
        b.release_all();
        const uint32_t h = n / 2;
        const int r1 = deft4cu_optimise_batch(in, in_len, h, flags, results);
        if (r1 && r1 != DEFT4CU_ERR_UNSUPPORTED) return r1;
        const int r2 = deft4cu_optimise_batch(in + h, in_len + h, n - h, flags, results + h);
        return r2 ? r2 : r1;
    }
    if (rc) {
        if (rc == DEFT4CU_ERR_UNSUPPORTED && b.infos.size() == n) {
            for (uint32_t i = 0; i < n; i++) { memset(&results[i], 0, sizeof results[i]); results[i].status = b.infos[i].status; }
        }
        return rc;
    }
    std::vector<uint8_t> sel(n, 1);
    rc = b.optimise(flags, sel);
    if (rc && rc != DEFT4CU_ERR_UNSUPPORTED) return rc;
    int rc2 = b.write();
    if (rc2) return rc2;
    rc2 = b.checksums();
    if (rc2) return rc2;
    rc2 = fill_results(b, results, true);
    return rc2 ? rc2 : rc;
}
int deft4cu_compress_batch(const uint8_t* const* in, const uint64_t* in_len, uint32_t n, uint32_t flags, uint32_t block_bytes,
                           deft4cu_result* results) {
    int rc = compress_block_bytes(&block_bytes);
    if (rc) return rc;
    rc = ensure_init();
    if (rc) return rc;
    Batch b;
    rc = b.upload(in, in_len, n);
    if (rc) return rc;
    rc = b.compress(block_bytes);
    if (rc == DEFT4CU_ERR_UNSUPPORTED && b.too_big && n > 1) {
        // more than 4 GiB of input: the list is compressed in two halves (streams never interact)
        b.release_all();
        const uint32_t h = n / 2;
        const int r1 = deft4cu_compress_batch(in, in_len, h, flags, block_bytes, results);
        if (r1 && r1 != DEFT4CU_ERR_UNSUPPORTED) return r1;
        const int r2 = deft4cu_compress_batch(in + h, in_len + h, n - h, flags, block_bytes, results + h);
        return r2 ? r2 : r1;
    }
    if (rc) {
        if (rc == DEFT4CU_ERR_UNSUPPORTED && b.infos.size() == n) {
            for (uint32_t i = 0; i < n; i++) { memset(&results[i], 0, sizeof results[i]); results[i].status = b.infos[i].status; }
        }
        return rc;
    }
    std::vector<uint8_t> sel(n, 1);
    rc = b.optimise(flags, sel);
    if (rc && rc != DEFT4CU_ERR_UNSUPPORTED) return rc;
    int rc2 = b.write();
    if (rc2) return rc2;
    rc2 = b.checksums();
    if (rc2) return rc2;
    rc2 = fill_results(b, results, true);
    return rc2 ? rc2 : rc;
}
void deft4cu_free_results(deft4cu_result* results, uint32_t n) {
    for (uint32_t i = 0; i < n; i++) { host_release(results[i].out); results[i].out = nullptr; }
}

// ---- facade -------------------------------------------------------------------------------------------------
int deft4cu_optimise_deflate_stream(const uint8_t* in, uint64_t len, int merge_blocks, uint8_t** out, uint64_t* out_len) {
    *out = nullptr;
    *out_len = 0;
    deft4cu_result r;
    memset(&r, 0, sizeof r);
    r.status = DEFT4CU_ERR_PARSE;
    int rc = deft4cu_optimise_batch(&in, &len, 1, merge_blocks ? DEFT4CU_MERGE_BLOCKS : 0, &r);
    // a parse failure or an unsupported stream keeps the caller's array (Deft.java:25-33); anything else is an error
    if (rc != DEFT4CU_OK && rc != DEFT4CU_ERR_UNSUPPORTED && rc != DEFT4CU_ERR_PARSE) { host_release(r.out); return rc; }
    if (r.status == ST_OK && r.saved_bits > 0) { *out = r.out; *out_len = r.out_len; }
    else host_release(r.out);
    return DEFT4CU_OK;
}
void deft4cu_free_buffer(uint8_t* p) { host_release(p); }
int64_t deft4cu_size_bits_fallback(const uint8_t* in, uint64_t len) {
    deft4cu_stream* s = nullptr;
    uint64_t c;
    if (deft4cu_stream_parse(in, len, &s, &c) != DEFT4CU_OK || !s) return (int64_t)len * 8;
    int64_t v = deft4cu_stream_size_bits(s);
    deft4cu_stream_free(s);
    return v;
}

// ---- device-resident batch (bench) -----------------------------------------------------------------------
int deft4cu_device_batch_create(const uint8_t* const* in, const uint64_t* in_len, uint32_t n, deft4cu_device_batch** out) {
    int rc = ensure_init();
    if (rc) return rc;
    auto b = std::make_shared<Batch>();
    rc = b->upload(in, in_len, n);
    if (rc) return rc;
    D4_CUDA_CHECK(cudaStreamSynchronize(b->cs));
    b->drop_stage();
    *out = new deft4cu_device_batch{b};
    return DEFT4CU_OK;
}
int deft4cu_device_batch_run(deft4cu_device_batch* db, uint32_t flags, uint64_t* launches, void* cuda_stream) {
    Batch& b = *db->batch;
    // run on the caller's stream when one is given (bench.py brackets the steps with events on that stream)
    b.cs = cuda_stream ? (cudaStream_t)cuda_stream : b.own_cs;
    b.launches = 0;
    int rc = b.parse();
    if (rc) return rc;
    std::vector<uint8_t> sel(b.n, 1);
    rc = b.optimise(flags, sel);
    if (rc && rc != DEFT4CU_ERR_UNSUPPORTED) return rc;
    int rc2 = b.write();
    if (rc2) return rc2;
    rc2 = b.checksums();
    if (rc2) return rc2;
    if (launches) *launches = b.launches;
    return rc;
}
int deft4cu_device_batch_fetch(deft4cu_device_batch* db, deft4cu_result* results) { return fill_results(*db->batch, results, true); }
int deft4cu_device_batch_timings(const deft4cu_device_batch* db, float* ms, uint32_t n) {
    for (uint32_t i = 0; i < n && i < 8; i++) ms[i] = db->batch->ms[i];
    return DEFT4CU_OK;
}
void deft4cu_device_batch_free(deft4cu_device_batch* db) { delete db; }

}  // extern "C"
