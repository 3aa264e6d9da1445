"""ctypes binding of libdeft4cu.so (the C ABI in include/deft4cu.h).

There is no CPU fallback: importing works without a GPU (so CPU-only tests can check the exported
symbols), but every compute call raises when the library or a CUDA device is missing.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DEFT4CU_LIB selects another build of the same ABI (tests use the small-pool stress build)
LIB_PATH = os.environ.get("DEFT4CU_LIB") or os.path.join(_HERE, "libdeft4cu.so")

OK, ERR_PARSE, ERR_WRITE, ERR_UNSUPPORTED, ERR_CUDA, ERR_ARG = 0, 1, 2, 3, 4, 5
MERGE_BLOCKS = 1


class Result(C.Structure):
    _fields_ = [("status", C.c_int32), ("consumed_bytes", C.c_uint64), ("saved_bits", C.c_int64),
                ("out", C.POINTER(C.c_uint8)), ("out_len", C.c_uint64), ("uncompressed_len", C.c_uint64),
                ("crc32", C.c_uint32), ("adler32", C.c_uint32), ("size_bits_in", C.c_int64),
                ("size_bits_out", C.c_int64)]


class BlockInfo(C.Structure):
    _fields_ = [("type", C.c_int32), ("size_bits", C.c_int64), ("position", C.c_int64),
                ("uncompressed_len", C.c_uint64), ("n_symbols", C.c_uint32), ("n_rle_pairs", C.c_uint32),
                ("num_litlen_lens", C.c_int32), ("num_dist_lens", C.c_int32), ("num_codelen_lens", C.c_int32),
                ("litlen_size_bits", C.c_int64), ("header_size_bits", C.c_int64)]


class FileResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("n_streams", C.c_uint32), ("saved_bits", C.c_int64),
                ("out", C.POINTER(C.c_uint8)), ("out_len", C.c_uint64), ("stream_saved", C.POINTER(C.c_int64)),
                ("stream_name", C.POINTER(C.c_char_p))]


# every symbol include/deft4cu.h declares: (restype, argtypes)
_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_U8PP = C.POINTER(C.c_char_p)
_U64P = C.POINTER(C.c_uint64)
SYMBOLS = {
    "deft4cu_init": (C.c_int, [C.c_int]),
    "deft4cu_last_error": (C.c_char_p, []),
    "deft4cu_version": (C.c_char_p, []),
    "deft4cu_optimise_batch": (C.c_int, [_U8PP, _U64P, C.c_uint32, C.c_uint32, C.POINTER(Result)]),
    "deft4cu_compress_batch": (C.c_int, [_U8PP, _U64P, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Result)]),
    "deft4cu_free_results": (None, [C.POINTER(Result), C.c_uint32]),
    "deft4cu_stream_parse": (C.c_int, [C.c_char_p, C.c_uint64, _PP, _U64P]),
    "deft4cu_stream_parse_batch": (C.c_int, [_U8PP, _U64P, C.c_uint32, _PP, C.POINTER(C.c_int32), _U64P]),
    "deft4cu_stream_compress_batch": (C.c_int, [_U8PP, _U64P, C.c_uint32, C.c_uint32, _PP, C.POINTER(C.c_int32)]),
    "deft4cu_stream_free": (None, [_P]),
    "deft4cu_stream_optimise": (C.c_int, [_P, C.c_uint32, C.POINTER(C.c_int64)]),
    "deft4cu_stream_optimise_batch": (C.c_int, [_PP, C.c_uint32, C.c_uint32, C.POINTER(C.c_int64)]),
    "deft4cu_stream_size_bits": (C.c_int64, [_P]),
    "deft4cu_stream_uncompressed_len": (C.c_uint64, [_P]),
    "deft4cu_stream_uncompressed": (C.c_int, [_P, C.c_char_p, C.c_uint64]),
    "deft4cu_stream_checksums": (C.c_int, [_P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "deft4cu_stream_write": (C.c_int, [_P, C.c_char_p, C.c_uint64, _U64P]),
    "deft4cu_stream_block_count": (C.c_uint32, [_P]),
    "deft4cu_stream_block_info": (C.c_int, [_P, C.c_uint32, C.POINTER(BlockInfo)]),
    "deft4cu_stream_block_symbols": (C.c_uint32, [_P, C.c_uint32, C.POINTER(C.c_int32), C.c_uint32]),
    "deft4cu_stream_block_rle_pairs": (C.c_uint32, [_P, C.c_uint32, C.POINTER(C.c_int32), C.c_uint32]),
    "deft4cu_stream_block_codelens": (C.c_uint32, [_P, C.c_uint32, C.c_int, C.POINTER(C.c_int32), C.c_uint32]),
    "deft4cu_optimise_deflate_stream": (C.c_int, [C.c_char_p, C.c_uint64, C.c_int, C.POINTER(C.POINTER(C.c_uint8)), _U64P]),
    "deft4cu_free_buffer": (None, [C.POINTER(C.c_uint8)]),
    "deft4cu_size_bits_fallback": (C.c_int64, [C.c_char_p, C.c_uint64]),
    "deft4cu_png_optimise_batch": (C.c_int, [_U8PP, _U64P, C.c_uint32, C.c_uint32, C.POINTER(FileResult)]),
    "deft4cu_zip_optimise_batch": (C.c_int, [_U8PP, _U64P, C.c_uint32, C.c_uint32, C.POINTER(FileResult)]),
    "deft4cu_gz_optimise_batch": (C.c_int, [_U8PP, _U64P, C.c_uint32, C.c_uint32, C.POINTER(FileResult)]),
    "deft4cu_zlib_optimise_batch": (C.c_int, [_U8PP, _U64P, C.c_uint32, C.c_uint32, C.POINTER(FileResult)]),
    "deft4cu_free_file_results": (None, [C.POINTER(FileResult), C.c_uint32]),
    "deft4cu_crc32": (C.c_uint32, [C.c_uint32, C.c_char_p, C.c_uint64]),
    "deft4cu_device_batch_create": (C.c_int, [_U8PP, _U64P, C.c_uint32, _PP]),
    "deft4cu_device_batch_run": (C.c_int, [_P, C.c_uint32, _U64P, _P]),
    "deft4cu_device_batch_fetch": (C.c_int, [_P, C.POINTER(Result)]),
    "deft4cu_device_batch_timings": (C.c_int, [_P, C.POINTER(C.c_float), C.c_uint32]),
    "deft4cu_device_batch_free": (None, [_P]),
    "deft4cu_debug_trace_begin": (C.c_int, [C.c_uint32]),
    "deft4cu_debug_trace_end": (C.c_int, [C.POINTER(C.c_int64), C.c_uint32, C.POINTER(C.c_uint32)]),
    "deft4cu_debug_prof": (C.c_int, [C.POINTER(C.c_uint64), C.c_uint32, C.c_int]),
    "deft4cu_debug_engine_launches": (C.c_uint64, []),
}

_lib = None
_inited = False


class Deft4cuError(RuntimeError):
    pass


def load():
    """dlopen the library and declare prototypes (works without a GPU)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Deft4cuError("libdeft4cu.so is not built (run __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def lib():
    """Library with an initialised CUDA device (LOCAL_RANK picks the GPU: one process per GPU)."""
    global _inited
    L = load()
    if not _inited:
        dev = int(os.environ.get("DEFT4CU_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        rc = L.deft4cu_init(dev)
        if rc != OK:
            raise Deft4cuError("deft4cu_init(%d) failed: %s (no CPU fallback)" % (dev, L.deft4cu_last_error().decode()))
        _inited = True
    return L


def last_error():
    return load().deft4cu_last_error().decode()


def make_ptr_arrays(buffers):
    """(char*[] , uint64[]) for a list of bytes objects; keeps references alive via the returned tuple."""
    n = len(buffers)
    ptrs = (C.c_char_p * max(n, 1))()
    lens = (C.c_uint64 * max(n, 1))()
    for i, b in enumerate(buffers):
        ptrs[i] = b
        lens[i] = len(b)
    return ptrs, lens
