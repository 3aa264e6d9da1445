"""deft4j_b200 — B200-native deflate stream optimiser: a drop-in for deft4j's `optimise -m NONE` path.

Host-side mirror of the reference API (DeflateStream, Deft, the container wrappers) over the C ABI of
libdeft4cu.so (include/deft4cu.h).  All deflate work runs in hand-written CUDA kernels for sm_100a;
there is no CPU fallback.
"""
from .deflate_stream import DeflateStream
from .deft import Deft, compress_batch, optimise_batch
from . import container

__all__ = ["DeflateStream", "Deft", "compress_batch", "optimise_batch", "container"]
