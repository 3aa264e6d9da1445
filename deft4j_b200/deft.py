"""Deft — mirror of the reference facade (base/Deft.java:16-54)."""
import ctypes as C

from . import _native as N


class Deft:
    @staticmethod
    def optimiseDeflateStream(original, mergeBlocks=True):
        """Deft.optimiseDeflateStream(byte[], boolean) (Deft.java:21-34): returns the SAME object when
        nothing was saved or the stream does not parse."""
        L = N.lib()
        out = C.POINTER(C.c_uint8)()
        out_len = C.c_uint64(0)
        data = bytes(original)
        rc = L.deft4cu_optimise_deflate_stream(data, len(data), 1 if mergeBlocks else 0, C.byref(out), C.byref(out_len))
        if rc != N.OK:
            raise N.Deft4cuError(N.last_error())
        if not out:
            return original
        try:
            return C.string_at(out, out_len.value)
        finally:
            L.deft4cu_free_buffer(out)

    @staticmethod
    def getSizeBitsFallback(deflateStream):  # Deft.java:48-54
        data = bytes(deflateStream)
        return N.lib().deft4cu_size_bits_fallback(data, len(data))


def optimise_batch(buffers, mergeBlocks=True):
    """Batch entry (deft4cu_optimise_batch): list of raw deflate streams -> list of dict results."""
    L = N.lib()
    n = len(buffers)
    ptrs, lens = N.make_ptr_arrays(buffers)
    res = (N.Result * max(n, 1))()
    rc = L.deft4cu_optimise_batch(ptrs, lens, n, N.MERGE_BLOCKS if mergeBlocks else 0, res)
    return _results(L, rc, res, n)


def compress_batch(buffers, mergeBlocks=True, block_bytes=0):
    """Compression entry (deft4cu_compress_batch): list of raw data buffers -> list of dict results like optimise_batch's,
    whose "out" is a raw deflate stream of the data.  block_bytes = 0 is the default block size (32768)."""
    L = N.lib()
    n = len(buffers)
    ptrs, lens = N.make_ptr_arrays(buffers)
    res = (N.Result * max(n, 1))()
    rc = L.deft4cu_compress_batch(ptrs, lens, n, N.MERGE_BLOCKS if mergeBlocks else 0, block_bytes, res)
    return _results(L, rc, res, n)


def _results(L, rc, res, n):
    if rc in (N.ERR_CUDA, N.ERR_ARG):
        raise N.Deft4cuError(N.last_error())
    out = []
    for i in range(n):
        r = res[i]
        out.append({
            "status": r.status, "consumed": r.consumed_bytes, "saved_bits": r.saved_bits,
            "out": C.string_at(r.out, r.out_len) if r.status == N.OK and r.out else None,
            "uncompressed_len": r.uncompressed_len, "crc32": r.crc32, "adler32": r.adler32,
            "size_bits_in": r.size_bits_in, "size_bits_out": r.size_bits_out,
        })
    L.deft4cu_free_results(res, n)
    return out
