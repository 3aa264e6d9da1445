/*
 * deft4cu.h — C ABI of the B200-native deflate stream optimiser (libdeft4cu.so).
 *
 * This is the drop-in boundary for the `deft4j optimise -m NONE` hot path: every entry point below
 * replaces one method of the reference's deft4j-base stream model (paths relative to
 * deft4j-base/src/main/java/com/github/NeRdTheNed/deft4j/).  Plain pointers and sizes only; no torch
 * types.  A Java facade binds these through Panama FFM (see INTEGRATION.md); the Python package
 * deft4j_b200 binds them through ctypes.
 *
 * All work (Huffman decode, LZ77 resolve, the block cost model / candidate enumerator, the bit writer)
 * runs in CUDA kernels on the selected device.  There is no CPU fallback: every call fails with
 * DEFT4CU_ERR_CUDA when no device is usable.
 *
 * Threading: calls on distinct handles may come from different host threads; one handle must not be
 * used concurrently.  The library owns all outputs until the matching free.
 */
#ifndef DEFT4CU_H
#define DEFT4CU_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* status codes */
#define DEFT4CU_OK 0
#define DEFT4CU_ERR_PARSE 1        /* DeflateStream.parse returned false (DeflateStream.java:105,109) */
#define DEFT4CU_ERR_WRITE 2        /* DeflateStream.write failed → IOException in asBytes (:652-660) */
#define DEFT4CU_ERR_UNSUPPORTED 3  /* input the reference accepts by accident (SURVEY.md H10) or that
                                      exceeds an internal limit; reported instead of emulated */
#define DEFT4CU_ERR_CUDA 4         /* no device / CUDA runtime error */
#define DEFT4CU_ERR_ARG 5

/* optimise flags */
#define DEFT4CU_MERGE_BLOCKS 1u    /* DeflateStream.optimise(boolean mergeBlocks) (:496) */

/* Library / device management.  deft4cu_init selects the CUDA device used by this process (one
 * process per GPU; multi-GPU runs shard streams across processes, SURVEY.md §8e). */
int         deft4cu_init(int device);
const char* deft4cu_last_error(void);
const char* deft4cu_version(void);

/* ------------------------------------------------------------------------------------------------
 * Batch entry — replaces `static DeflateFilesContainer.optimise(List<DeflateStream>, boolean)`
 * (deft4j-container/.../DeflateFilesContainer.java:18-43) fused with parse and write: n independent
 * raw deflate streams in, n optimised streams out.
 * ---------------------------------------------------------------------------------------------- */
typedef struct deft4cu_result {
    int32_t  status;            /* DEFT4CU_* */
    uint64_t consumed_bytes;    /* bytes of input consumed by parse (containers read trailers after it) */
    int64_t  saved_bits;        /* return value of DeflateStream.optimise (:565) */
    uint8_t* out;               /* DeflateStream.asBytes() (:652-660); library-owned */
    uint64_t out_len;
    uint64_t uncompressed_len;  /* getUncompressedData().length (:159-169) */
    uint32_t crc32;             /* CRC-32 of the uncompressed data (GZFile.java:130-145)  */
    uint32_t adler32;           /* Adler-32 of the uncompressed data (ZLibFile.java:42-51) */
    int64_t  size_bits_in;      /* getSizeBits() before optimise (:171-182) */
    int64_t  size_bits_out;     /* getSizeBits() after optimise */
} deft4cu_result;

int  deft4cu_optimise_batch(const uint8_t* const* in, const uint64_t* in_len, uint32_t n, uint32_t flags,
                            deft4cu_result* results);
void deft4cu_free_results(deft4cu_result* results, uint32_t n);

/* ------------------------------------------------------------------------------------------------
 * Compression — raw bytes in, optimised deflate out.  The device cuts every input into blocks of block_bytes
 * (0: 32768; otherwise 256..65535, else DEFT4CU_ERR_ARG), finds LZ77 matches with a lazy parse and models the
 * result as a fixed-coded stream F (the rule: deft4j_b200/csrc/lzrule.cuh), which the optimiser then entropy-codes.
 * size_bits_in = bits of F, saved_bits = what optimise saved against F, consumed_bytes = uncompressed_len = input
 * length.  flags honours DEFT4CU_MERGE_BLOCKS.  The output is this library's own; it is not any CPU compressor's.
 * ---------------------------------------------------------------------------------------------- */
int  deft4cu_compress_batch(const uint8_t* const* in, const uint64_t* in_len, uint32_t n, uint32_t flags,
                            uint32_t block_bytes, deft4cu_result* results);

/* ------------------------------------------------------------------------------------------------
 * Handle API — mirrors the DeflateStream object (base/deflate/DeflateStream.java)
 * ---------------------------------------------------------------------------------------------- */
typedef struct deft4cu_stream deft4cu_stream;

/* DeflateStream.parse(byte[] / InputStream) (:63-126).  *consumed = bytes consumed. */
int      deft4cu_stream_parse(const uint8_t* data, uint64_t len, deft4cu_stream** out, uint64_t* consumed);
/* several streams parsed together (one launch); handles[i] is NULL where status[i] != OK */
int      deft4cu_stream_parse_batch(const uint8_t* const* data, const uint64_t* len, uint32_t n,
                                    deft4cu_stream** handles, int32_t* status, uint64_t* consumed);
/* handles of raw inputs compressed on the device (deft4cu_compress_batch's first step); writing one before optimise
 * gives the fixed-coded stream F.  handles[i] is NULL where status[i] != OK. */
int      deft4cu_stream_compress_batch(const uint8_t* const* data, const uint64_t* len, uint32_t n, uint32_t block_bytes,
                                       deft4cu_stream** handles, int32_t* status);
void     deft4cu_stream_free(deft4cu_stream* s);
/* DeflateStream.optimise(boolean) (:496-566) */
int      deft4cu_stream_optimise(deft4cu_stream* s, uint32_t flags, int64_t* saved_bits);
/* batched: optimise many parsed streams in the same launches (DeflateFilesContainer.java:18-43) */
int      deft4cu_stream_optimise_batch(deft4cu_stream* const* s, uint32_t n, uint32_t flags, int64_t* saved_bits);
/* DeflateStream.getSizeBits() (:171-182) */
int64_t  deft4cu_stream_size_bits(const deft4cu_stream* s);
/* DeflateStream.getUncompressedData() (:159-169): length, copy-out, and device-computed checksums */
uint64_t deft4cu_stream_uncompressed_len(const deft4cu_stream* s);
int      deft4cu_stream_uncompressed(const deft4cu_stream* s, uint8_t* dst, uint64_t cap);
int      deft4cu_stream_checksums(const deft4cu_stream* s, uint32_t* crc32, uint32_t* adler32);
/* DeflateStream.write / asBytes (:128-145,652-660): returns needed length in *len; copies when cap fits */
int      deft4cu_stream_write(const deft4cu_stream* s, uint8_t* dst, uint64_t cap, uint64_t* len);
/* printBlockInfo (:35-51) and model inspection used by the parity tests */
typedef struct deft4cu_block_info {
    int32_t  type;              /* DeflateBlockType ordinal: 0 STORED, 1 FIXED, 2 DYNAMIC */
    int64_t  size_bits;         /* getSizeBits(pos) without the 3 header bits */
    int64_t  position;          /* bit position of the block header in the (re)written stream */
    uint64_t uncompressed_len;
    uint32_t n_symbols;         /* litlens.size() after optimisation (replaced matches count as literals) */
    uint32_t n_rle_pairs;
    int32_t  num_litlen_lens, num_dist_lens, num_codelen_lens;
    int64_t  litlen_size_bits, header_size_bits;
} deft4cu_block_info;
uint32_t deft4cu_stream_block_count(const deft4cu_stream* s);
int      deft4cu_stream_block_info(const deft4cu_stream* s, uint32_t block, deft4cu_block_info* out);
/* symbols of a block as {dist, litlen, edgecase} triples (LitLen.java:29-47); returns count */
uint32_t deft4cu_stream_block_symbols(const deft4cu_stream* s, uint32_t block, int32_t* dst, uint32_t cap_syms);
/* header RLE pairs {dist, sym}; returns count */
uint32_t deft4cu_stream_block_rle_pairs(const deft4cu_stream* s, uint32_t block, int32_t* dst, uint32_t cap);
/* code length tables: which = 0 litlen, 1 dist, 2 codelen; returns length */
uint32_t deft4cu_stream_block_codelens(const deft4cu_stream* s, uint32_t block, int which, int32_t* dst, uint32_t cap);

/* ------------------------------------------------------------------------------------------------
 * Facade — Deft.optimiseDeflateStream(byte[], boolean) (base/Deft.java:21-34): returns 0 and a
 * library-owned buffer when bits were saved; returns 0 with *out == NULL when the caller should keep
 * its own array (nothing saved or parse failure), exactly like the reference returns `original`.
 * ---------------------------------------------------------------------------------------------- */
int  deft4cu_optimise_deflate_stream(const uint8_t* in, uint64_t len, int merge_blocks, uint8_t** out, uint64_t* out_len);
void deft4cu_free_buffer(uint8_t* p);
/* Deft.getSizeBitsFallback (Deft.java:48-54) */
int64_t deft4cu_size_bits_fallback(const uint8_t* in, uint64_t len);

/* ------------------------------------------------------------------------------------------------
 * File front-end for PNG / APNG — replaces, for a LIST of files, PNGFile.read (deft4j-container/.../
 * container/PNGFile.java:574-605, chunk reader :162-215, PNGChunkHelper :413-572), the container's
 * optimise (DeflateFilesContainer.java:18-43 over getDeflateStreams(), PNGFile.java:376-389) and
 * PNGFile.write (:391-411 with syncStreams :262-369).  The chunk model runs on host threads; the IDAT /
 * fdAT / zTXt / iCCP / iTXt zlib streams of all files are ONE device batch.
 * status: OK; ERR_PARSE where PNGFile.read returns false; ERR_WRITE where write() throws; ERR_UNSUPPORTED
 * where a stream hit an internal limit.  Streams are listed in getDeflateStreams() order.
 * ---------------------------------------------------------------------------------------------- */
typedef struct deft4cu_file_result {
    int32_t  status;
    uint32_t n_streams;          /* getDeflateStreams().size() */
    int64_t  saved_bits;         /* return value of DeflateFilesContainer.optimise (:18-43) */
    uint8_t* out;                /* PNGFile.write(); library-owned */
    uint64_t out_len;
    int64_t* stream_saved;       /* n_streams entries: bits saved per stream */
    char**   stream_name;        /* n_streams NUL-terminated names: "IDAT chunk", "fdAT chunk 2", "zTXt chunk"
                                    (PNGFile.java:441,:458,:536); the entry's file name for ZIP (ZipFile.java:100-124) */
} deft4cu_file_result;
int  deft4cu_png_optimise_batch(const uint8_t* const* files, const uint64_t* lens, uint32_t n, uint32_t flags,
                                deft4cu_file_result* results);
/* The same for ZIP archives — ZipFile.read (deft4j-container/.../container/ZipFile.java:82-127: entries with method 8
 * become streams, in local-file order), optimise, ZipFile.write (:46-79) through RecalculatingZipWriter
 * (container/lljzip/RecalculatingZipWriter.java:23-136).  The archive reader restates the standard strategy of the
 * un-vendored lljzip 2.3.0 (parity unpinned).  ERR_PARSE: no end record / Zip64 / no local headers / an entry that does
 * not parse; ERR_WRITE: a central directory entry without its local header. */
int  deft4cu_zip_optimise_batch(const uint8_t* const* files, const uint64_t* lens, uint32_t n, uint32_t flags,
                                deft4cu_file_result* results);
/* The same for gzip members — GZFile.read (deft4j-container/.../container/GZFile.java:42-87), optimise, GZFile.write
 * (:92-152: header fields written back, FCOMMENT without its NUL, CRC-32 and ISIZE recalculated from the decoded data —
 * here: taken from the device) — and for zlib streams — ZLibFile.read (container/ZLibFile.java:59-95), ZLibFile.write
 * (:33-57, Adler-32 recalculated).  One stream per file, named after FNAME (gzip) or "unnamed stream". */
int  deft4cu_gz_optimise_batch(const uint8_t* const* files, const uint64_t* lens, uint32_t n, uint32_t flags,
                               deft4cu_file_result* results);
int  deft4cu_zlib_optimise_batch(const uint8_t* const* files, const uint64_t* lens, uint32_t n, uint32_t flags,
                                 deft4cu_file_result* results);
void deft4cu_free_file_results(deft4cu_file_result* results, uint32_t n);
/* java.util.zip.CRC32 as the chunk writer uses it (PNGFile.java:140-158); crc = 0 starts a new checksum */
uint32_t deft4cu_crc32(uint32_t crc, const uint8_t* data, uint64_t len);

/* ------------------------------------------------------------------------------------------------
 * Device-resident benchmarking entry (bench.py `value`): inputs already in HBM.  Times nothing itself;
 * runs parse → optimise → write for a batch whose input bytes live at d_in (device pointer) and leaves
 * the output on the device.  Kernel launch counts are returned for the `gpu_launches` bench key.
 * ---------------------------------------------------------------------------------------------- */
typedef struct deft4cu_device_batch deft4cu_device_batch;
int  deft4cu_device_batch_create(const uint8_t* const* in, const uint64_t* in_len, uint32_t n, deft4cu_device_batch** out);
int  deft4cu_device_batch_run(deft4cu_device_batch* b, uint32_t flags, uint64_t* launches, void* cuda_stream);
int  deft4cu_device_batch_fetch(deft4cu_device_batch* b, deft4cu_result* results); /* D2H of the last run */
/* per-kernel-family device time of the last run in ms (CUDA events on the run's stream):
 * [0] parse/count [1] emit [2] lz77 [3] optimise (candidate engine) [4] merge [5] write [6] checksums */
int  deft4cu_device_batch_timings(const deft4cu_device_batch* b, float* ms, uint32_t n);
void deft4cu_device_batch_free(deft4cu_device_batch* b);

/* ------------------------------------------------------------------------------------------------
 * Parity-debug instrumentation (tests and scripts only): while armed, the candidate enumerator logs every
 * candidate the selection callback of DeflateStream.optimiseBlock (DeflateStream.java:349-368) compares, as
 * {candidate index within the call, size in bits} pairs ({-1, incumbent size} opens each call), so a
 * divergence from the oracle can be located.  Meaningful for one block at a time.
 * ---------------------------------------------------------------------------------------------- */
int  deft4cu_debug_trace_begin(uint32_t cap_pairs);
int  deft4cu_debug_trace_end(int64_t* dst_pairs, uint32_t cap_pairs, uint32_t* n_pairs);
/* Launches of the candidate engine kernel since the library was loaded: DeflateFilesContainer.optimise's stream list
 * (DeflateFilesContainer.java:18-43) is meant to cost one. */
uint64_t deft4cu_debug_engine_launches(void);
/* Engine phase cycle counters (only in a -DD4_PROF build of the library; DEFT4CU_ERR_ARG otherwise):
 * dst[c] = cycles, dst[32 + c] = calls for phase category c (engine.cuh PR_*). */
int  deft4cu_debug_prof(uint64_t* dst, uint32_t n, int reset);

#ifdef __cplusplus
}
#endif
#endif
