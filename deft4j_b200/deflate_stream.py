"""DeflateStream — host-side mirror of deft4j-base's DeflateStream (base/deflate/DeflateStream.java),
backed by the CUDA library through the handle API of include/deft4cu.h.

Method names, argument meaning and failure behaviour follow the reference: parse/write return bool,
asBytes raises IOError, optimise returns the number of bits saved.
"""
import ctypes as C

from . import _native as N

_TYPE_NAMES = ["STORED", "FIXED", "DYNAMIC"]


class DeflateStream:
    DEFAULT_NAME = "unnamed stream"  # DeflateStream.java:19

    def __init__(self, name=None):
        self.name = name if name is not None else self.DEFAULT_NAME
        self._h = None
        self.consumed = 0

    def __del__(self):
        try:
            if self._h is not None:
                N.load().deft4cu_stream_free(self._h)
                self._h = None
        except Exception:
            pass

    def getName(self):
        return self.name

    def setName(self, name):
        self.name = name

    # -- parse(byte[] | InputStream) (:63-126) ----------------------------------------------------
    def parse(self, src):
        from .container._io import ByteReader
        data = src.remaining() if isinstance(src, ByteReader) else bytes(src)
        L = N.lib()
        h = C.c_void_p()
        consumed = C.c_uint64(0)
        rc = L.deft4cu_stream_parse(data, len(data), C.byref(h), C.byref(consumed))
        if rc in (N.ERR_CUDA, N.ERR_ARG):
            raise N.Deft4cuError(N.last_error())
        self.consumed = consumed.value
        if isinstance(src, ByteReader):
            src.pos += consumed.value
        if rc != N.OK or not h.value:
            return False
        self._h = h
        return True

    @classmethod
    def parse_batch(cls, buffers, names=None):
        """Parse many streams in one device batch; returns a list of DeflateStream (None where parse failed)."""
        L = N.lib()
        n = len(buffers)
        ptrs, lens = N.make_ptr_arrays(buffers)
        handles = (C.c_void_p * max(n, 1))()
        status = (C.c_int32 * max(n, 1))()
        consumed = (C.c_uint64 * max(n, 1))()
        rc = L.deft4cu_stream_parse_batch(ptrs, lens, n, handles, status, consumed)
        if rc != N.OK:
            raise N.Deft4cuError(N.last_error())
        out = []
        for i in range(n):
            if status[i] == N.OK and handles[i]:
                s = cls(names[i] if names else None)
                s._h = C.c_void_p(handles[i])
                s.consumed = consumed[i]
                out.append(s)
            else:
                out.append(None)
        return out

    @classmethod
    def compress_batch(cls, buffers, names=None, block_bytes=0):
        """Compress raw data buffers on the device (deft4cu_stream_compress_batch); returns a list of DeflateStream (None
        where a buffer was refused) whose model is the fixed-coded stream of the data, ready for optimise."""
        L = N.lib()
        n = len(buffers)
        ptrs, lens = N.make_ptr_arrays(buffers)
        handles = (C.c_void_p * max(n, 1))()
        status = (C.c_int32 * max(n, 1))()
        rc = L.deft4cu_stream_compress_batch(ptrs, lens, n, block_bytes, handles, status)
        if rc != N.OK:
            raise N.Deft4cuError(N.last_error())
        out = []
        for i in range(n):
            if status[i] == N.OK and handles[i]:
                s = cls(names[i] if names else None)
                s._h = C.c_void_p(handles[i])
                s.consumed = len(buffers[i])
                out.append(s)
            else:
                out.append(None)
        return out

    # -- optimise(boolean mergeBlocks) (:496-566) -------------------------------------------------
    def optimise(self, mergeBlocks=True):
        return self.optimise_batch([self], mergeBlocks)[0]

    @staticmethod
    def optimise_batch(streams, mergeBlocks=True):
        """DeflateFilesContainer.optimise's loop (DeflateFilesContainer.java:18-43) as one device batch."""
        L = N.lib()
        n = len(streams)
        hs = (C.c_void_p * max(n, 1))(*[s._h for s in streams])
        saved = (C.c_int64 * max(n, 1))()
        rc = L.deft4cu_stream_optimise_batch(hs, n, N.MERGE_BLOCKS if mergeBlocks else 0, saved)
        if rc != N.OK:
            raise N.Deft4cuError("optimise failed (%d): %s" % (rc, N.last_error()))
        return [saved[i] for i in range(n)]

    def getSizeBits(self):  # :171-182
        return N.lib().deft4cu_stream_size_bits(self._h)

    def getUncompressedData(self):  # :159-169
        L = N.lib()
        n = L.deft4cu_stream_uncompressed_len(self._h)
        buf = C.create_string_buffer(n if n else 1)
        rc = L.deft4cu_stream_uncompressed(self._h, buf, n)
        if rc != N.OK:
            raise N.Deft4cuError(N.last_error())
        return buf.raw[:n]

    def getChecksums(self):
        """(crc32, adler32, length) of the uncompressed data, computed on the device."""
        L = N.lib()
        crc, ad = C.c_uint32(), C.c_uint32()
        rc = L.deft4cu_stream_checksums(self._h, C.byref(crc), C.byref(ad))
        if rc != N.OK:
            raise N.Deft4cuError(N.last_error())
        return crc.value, ad.value, L.deft4cu_stream_uncompressed_len(self._h)

    def write(self):
        """write(OutputStream) (:128-145): returns the bytes, or None when the reference would return false."""
        L = N.lib()
        need = C.c_uint64(0)
        rc = L.deft4cu_stream_write(self._h, None, 0, C.byref(need))
        if rc in (N.ERR_CUDA, N.ERR_ARG):
            raise N.Deft4cuError(N.last_error())
        if rc != N.OK:
            return None
        buf = C.create_string_buffer(need.value if need.value else 1)
        rc = L.deft4cu_stream_write(self._h, buf, need.value, C.byref(need))
        if rc != N.OK:
            return None
        return buf.raw[:need.value]

    def asBytes(self):  # :652-660
        out = self.write()
        if out is None:
            raise IOError("Could not write deflate stream to bytes")
        return out

    # -- model inspection ----------------------------------------------------------------------------
    def blockCount(self):
        return N.lib().deft4cu_stream_block_count(self._h)

    def blockInfo(self, i):
        bi = N.BlockInfo()
        if N.lib().deft4cu_stream_block_info(self._h, i, C.byref(bi)) != N.OK:
            raise IndexError(i)
        return bi

    def blockSymbols(self, i):
        n = self.blockInfo(i).n_symbols
        arr = (C.c_int32 * (3 * max(n, 1)))()
        N.lib().deft4cu_stream_block_symbols(self._h, i, arr, n)
        return [(arr[3 * k], arr[3 * k + 1], arr[3 * k + 2]) for k in range(n)]

    def blockRlePairs(self, i):
        arr = (C.c_int32 * 640)()
        n = N.lib().deft4cu_stream_block_rle_pairs(self._h, i, arr, 320)
        return [(arr[2 * k], arr[2 * k + 1]) for k in range(n)]

    def blockCodelens(self, i, which):
        arr = (C.c_int32 * 320)()
        n = N.lib().deft4cu_stream_block_codelens(self._h, i, which, arr, 320)
        return list(arr[:n])

    def printBlockInfo(self):  # :35-51
        s = ""
        n = self.blockCount()
        for i in range(n):
            bi = self.blockInfo(i)
            s += "\nBlock %d position %d size %d type %s" % (i, bi.position, bi.size_bits + 3, _TYPE_NAMES[bi.type])
        return "Stream name: " + self.name + "\nBlock info:" + s + "\nTotal blocks: %d" % n
