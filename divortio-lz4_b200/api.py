"""Host-side mirror of the reference's block/frame interface over the C ABI (include/dlz4_b200.h).

The reference is JavaScript and no JS engine exists in this image, so the host side above the C ABI is
Python with the reference's names, argument order, defaults and error text:

  compressBlock(src, output, srcStart, srcLen, hashTable, outputOffset)      src/block/blockCompress.js:31
  decompressBlock(input, inputOffset, inputSize, output, outputOffset, dict) src/block/blockDecompress.js:30
  compressBuffer(input, dictionary, maxBlockSize, blockIndependence,
                 contentChecksum, addContentSize, outputBuffer)              src/buffer/bufferCompress.js:100
  decompressBuffer(input, dictionary, verifyChecksum)                        src/buffer/bufferDecompress.js:51
  xxHash32(input, seed)                                                      src/xxhash32/xxhash32.js:21
  LZ4.compressRaw / decompressRaw / compress / decompress                    src/lz4.js:32-35

plus the batched entry points the frame loops use (compress_blocks / decompress_blocks / xxh32_batch) and
their device-pointer forms.  Everything runs on the GPU through libdlz4_b200.so; there is no CPU fallback and
importing or calling without the built library / a CUDA device raises.
"""
import ctypes as C
import json
import os

import numpy as np

__all__ = [
    "LZ4", "LZ4Error", "Context", "default_context", "compressBlock", "decompressBlock", "compressBuffer",
    "decompressBuffer", "xxHash32", "compress_blocks", "decompress_blocks", "xxh32_batch", "compress_bound",
    "frame_bound", "shard_range", "ensureBuffer", "lib", "LIB_PATH", "WARM_NONE", "WARM_JENKINS", "WARM_TABLE",
    "HIST_RAW", "HIST_FRAME", "frame_info", "decompressFrames", "XXHash32", "chain_compress", "compressBuffers",
    "decompressBuffers",
]

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DLZ4_LIB") or os.path.join(_HERE, "csrc", "libdlz4_b200.so")

WARM_NONE, WARM_JENKINS, WARM_TABLE = 0, 1, 2
HIST_RAW, HIST_FRAME = 0, 1
E_CUDA = 30
E_BAD_VERSION = 6
E_DICT_OOB = 4
E_BAD_MAGIC = 5
E_CONTENT_CHECKSUM = 7


class LZ4Error(Exception):
    """Carries the reference's exception text ("LZ4: Malformed Input", ...) and the numeric status."""

    def __init__(self, status, message):
        super().__init__(message)
        self.status = status


class FrameInfo(C.Structure):
    _fields_ = [("content_size", C.c_uint64), ("max_decoded", C.c_uint64), ("nblocks", C.c_uint32),
                ("block_max_size", C.c_uint32), ("flg", C.c_uint8), ("bd", C.c_uint8), ("has_content_size", C.c_uint8),
                ("has_content_checksum", C.c_uint8), ("has_block_checksum", C.c_uint8), ("has_dict_id", C.c_uint8),
                ("block_independence", C.c_uint8), ("pad", C.c_uint8), ("dict_id", C.c_uint32), ("version", C.c_int32),
                ("frame_bytes", C.c_uint64)]


class Xxh32State(C.Structure):
    _fields_ = [("v", C.c_uint32 * 4), ("total", C.c_uint64), ("mem", C.c_uint8 * 16), ("memsize", C.c_uint32), ("seed", C.c_uint32)]


class FrameOpts(C.Structure):
    _fields_ = [("max_block_size", C.c_uint32), ("block_independence", C.c_int32), ("content_checksum", C.c_int32),
                ("add_content_size", C.c_int32), ("block_checksum", C.c_int32)]


_lib = None


def lib():
    """Loads libdlz4_b200.so.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libdlz4_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                           "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, u32, u64, i32, i64 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int32, C.c_int64
    sig = {
        "dlz4_init": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "dlz4_shutdown": (None, [vp]),
        "dlz4_strerror": (C.c_char_p, [C.c_int]),
        "dlz4_last_error": (C.c_char_p, [vp]),
        "dlz4_launch_count": (u64, [vp]),
        "dlz4_last_kernel_ms": (C.c_float, [vp]),
        "dlz4_kernel_probe": (C.c_int, [vp, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
        "dlz4_segment_stats": (None, [vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
        "dlz4_pinned_alloc": (vp, [u64]),
        "dlz4_pinned_free": (None, [vp]),
        "dlz4_host_register": (C.c_int, [vp, u64]),
        "dlz4_host_unregister": (C.c_int, [vp]),
        "dlz4_compress_bound": (u64, [u64]),
        "dlz4_frame_bound": (u64, [u64]),
        "dlz4_shard_range": (None, [u64, u32, u32, C.POINTER(u64), C.POINTER(u64)]),
        "dlz4_compress_blocks_dev": (C.c_int, [vp, vp, vp, vp, u32, u32, vp, u32, C.c_int, vp, vp, vp, vp, vp]),
        "dlz4_compress_blocks": (C.c_int, [vp, vp, u64, vp, vp, u32, vp, u32, C.c_int, vp, vp, u64, vp, vp]),
        "dlz4_decompress_blocks_dev": (C.c_int, [vp, vp, vp, vp, u32, vp, vp, vp, vp, u32, C.c_int, vp, vp, vp]),
        "dlz4_decompress_blocks": (C.c_int, [vp, vp, u64, vp, vp, u32, vp, u64, vp, vp, vp, u32, C.c_int, vp, vp]),
        "dlz4_compress_block": (C.c_int, [vp, vp, u64, i32, i32, vp, vp, u64, i32, C.POINTER(i32)]),
        "dlz4_decompress_block": (C.c_int, [vp, vp, u64, i64, i64, vp, u64, i64, vp, u64, C.POINTER(i64)]),
        "dlz4_xxh32_batch_dev": (C.c_int, [vp, vp, vp, vp, u32, u32, vp, vp]),
        "dlz4_xxh32_stream_dev": (C.c_int, [vp, vp, u64, u32, vp, vp]),
        "dlz4_xxh32": (C.c_int, [vp, vp, u64, u32, C.POINTER(u32)]),
        "dlz4_xxh32_async": (C.c_int, [vp, C.c_int, vp, u64, u32]),
        "dlz4_xxh32_wait": (C.c_int, [vp, C.c_int, C.POINTER(u32)]),
        "dlz4_xxh32_batch": (C.c_int, [vp, vp, u64, vp, vp, u32, u32, vp]),
        "dlz4_frame_compress": (C.c_int, [vp, vp, u64, vp, u64, C.POINTER(FrameOpts), vp, u64, C.POINTER(u64)]),
        "dlz4_frame_info": (C.c_int, [vp, u64, C.POINTER(FrameInfo)]),
        "dlz4_frame_decompress": (C.c_int, [vp, vp, u64, vp, u64, u32, vp, u64, C.POINTER(u64)]),
        "dlz4_frame_pack_dev": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, u32, C.c_int, vp, vp, vp]),
        "dlz4_frame_decompress_ex": (C.c_int, [vp, vp, u64, vp, u64, u32, vp, u64, C.POINTER(u64), vp]),
        "dlz4_frames_decompress": (C.c_int, [vp, vp, u64, vp, u64, u32, vp, u64, C.POINTER(u64), C.POINTER(u32)]),
        "dlz4_frames_info": (C.c_int, [vp, u64, C.POINTER(u64), C.POINTER(u32)]),
        "dlz4_xxh32_reset": (None, [C.POINTER(Xxh32State), u32]),
        "dlz4_xxh32_update": (C.c_int, [vp, C.POINTER(Xxh32State), vp, u64]),
        "dlz4_xxh32_digest": (u32, [C.POINTER(Xxh32State)]),
        "dlz4_chain_compress": (C.c_int, [vp, vp, u64, i32, i32, i32, vp, vp, u64, vp]),
        "dlz4_stream_blocks": (C.c_int, [vp, vp, u64, vp, u64, i32, i32, i32, C.c_int, vp, vp, u64, C.POINTER(u64), vp]),
        "dlz4_frame_body_compress": (C.c_int, [vp, vp, u64, u32, C.c_int, C.POINTER(u64)]),
        "dlz4_frame_body_fetch": (C.c_int, [vp, vp, u64]),
        "dlz4_frame_header": (C.c_size_t, [C.POINTER(FrameOpts), u64, C.c_int, u32, vp]),
        "dlz4_frame_decompress_range": (C.c_int, [vp, vp, u64, u32, u32, vp, u64, u32, vp, u64, C.POINTER(u64), vp]),
        "dlz4_xxh32_update_resident": (C.c_int, [vp, C.POINTER(Xxh32State), C.c_int]),
        "dlz4_frames_compress_batch_dev": (C.c_int, [vp, vp, vp, vp, u32, u32, vp, u32, C.POINTER(FrameOpts), vp, u64, vp, vp]),
        "dlz4_frames_compress_batch": (C.c_int, [vp, vp, u64, vp, vp, u32, vp, u32, C.POINTER(FrameOpts), vp, u64, vp]),
        "dlz4_frames_batch_info_dev": (C.c_int, [vp, vp, vp, vp, u32, vp, vp, vp]),
        "dlz4_frames_batch_info": (C.c_int, [vp, vp, u64, vp, vp, u32, vp, vp]),
        "dlz4_frames_decompress_batch_dev": (C.c_int, [vp, vp, vp, vp, u32, vp, u32, u32, vp, vp, vp, vp, vp, vp]),
        "dlz4_frames_decompress_batch": (C.c_int, [vp, vp, u64, vp, vp, u32, vp, u32, u32, vp, u64, vp, vp, vp, vp]),
        "dlz4_frame_compress_dev": (C.c_int, [vp, vp, u64, vp, u64, C.POINTER(FrameOpts), vp, u64, C.POINTER(u64), vp]),
        "dlz4_frame_info_dev": (C.c_int, [vp, vp, u64, C.POINTER(FrameInfo), vp]),
        "dlz4_frame_decompress_dev": (C.c_int, [vp, vp, u64, vp, u64, u32, vp, u64, C.POINTER(u64), vp]),
        "dlz4_frames_compress_dev": (C.c_int, [vp, vp, u64, u64, vp, u64, C.POINTER(FrameOpts), vp, u64, vp, C.POINTER(u64),
                                               C.POINTER(u32), vp]),
        "dlz4_frames_info_dev": (C.c_int, [vp, vp, u64, C.POINTER(u64), C.POINTER(u32), vp]),
        "dlz4_frames_decompress_dev": (C.c_int, [vp, vp, u64, vp, u64, u32, vp, u64, C.POINTER(u64), C.POINTER(u32), vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "dlz4_init", "dlz4_shutdown", "dlz4_strerror", "dlz4_last_error", "dlz4_launch_count", "dlz4_last_kernel_ms", "dlz4_kernel_probe", "dlz4_segment_stats",
    "dlz4_pinned_alloc", "dlz4_pinned_free", "dlz4_host_register", "dlz4_host_unregister", "dlz4_compress_bound", "dlz4_frame_bound", "dlz4_shard_range",
    "dlz4_compress_blocks_dev", "dlz4_compress_blocks", "dlz4_decompress_blocks_dev", "dlz4_decompress_blocks",
    "dlz4_compress_block", "dlz4_decompress_block", "dlz4_xxh32_batch_dev", "dlz4_xxh32_stream_dev", "dlz4_xxh32", "dlz4_xxh32_async", "dlz4_xxh32_wait",
    "dlz4_xxh32_batch", "dlz4_frame_compress", "dlz4_frame_info", "dlz4_frame_decompress", "dlz4_frame_pack_dev", "dlz4_frames_decompress", "dlz4_frames_info", "dlz4_frame_decompress_ex", "dlz4_xxh32_reset", "dlz4_xxh32_update", "dlz4_xxh32_digest",
    "dlz4_chain_compress", "dlz4_stream_blocks", "dlz4_frame_body_compress", "dlz4_frame_body_fetch", "dlz4_frame_header", "dlz4_frame_decompress_range",
    "dlz4_xxh32_update_resident", "dlz4_frames_compress_batch_dev", "dlz4_frames_compress_batch", "dlz4_frames_batch_info_dev",
    "dlz4_frames_batch_info", "dlz4_frames_decompress_batch_dev", "dlz4_frames_decompress_batch", "dlz4_frame_compress_dev",
    "dlz4_frame_info_dev", "dlz4_frame_decompress_dev", "dlz4_frames_compress_dev", "dlz4_frames_info_dev", "dlz4_frames_decompress_dev",
]


def ensureBuffer(x):
    """src/shared/lz4Util.js:13-33 -- String (UTF-8) / bytes-like / array of numbers / object (JSON) -> uint8 array."""
    if isinstance(x, np.ndarray):
        if x.dtype != np.uint8:
            x = x.view(np.uint8)
        return np.ascontiguousarray(x).reshape(-1)
    if isinstance(x, str):
        return np.frombuffer(x.encode("utf-8"), dtype=np.uint8)
    if isinstance(x, (bytes, bytearray, memoryview)):
        return np.frombuffer(x, dtype=np.uint8)
    if isinstance(x, (list, tuple)):
        return np.asarray(x, dtype=np.int64).astype(np.uint8)
    if isinstance(x, dict):
        return np.frombuffer(json.dumps(x, separators=(",", ":")).encode("utf-8"), dtype=np.uint8)
    raise TypeError("LZ4: Input must be a String, ArrayBuffer, View, Array or Object")


def _ptr(a):
    return a.ctypes.data if a is not None and a.size else None


class Context(object):
    """One per process and GPU: owns a CUDA stream and reusable device scratch (dlz4_ctx)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        L = lib()
        st = L.dlz4_init(int(device), C.byref(self._h))
        if st != 0:
            msg = L.dlz4_last_error(self._h).decode() if self._h else ""
            if self._h:
                L.dlz4_shutdown(self._h)
                self._h = C.c_void_p()
            raise RuntimeError("dlz4_init(device=%d) failed: %s -- a CUDA device is required, there is no CPU fallback"
                               % (device, msg))
        self.device = device

    @property
    def handle(self):
        return self._h

    def close(self):
        if self._h:
            lib().dlz4_shutdown(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, status, extra=""):
        if status == 0:
            return
        L = lib()
        if status == E_CUDA:
            raise RuntimeError("dlz4 CUDA failure: " + L.dlz4_last_error(self._h).decode())
        raise LZ4Error(status, L.dlz4_strerror(status).decode() + extra)

    @property
    def launch_count(self):
        return int(lib().dlz4_launch_count(self._h))

    @property
    def last_kernel_ms(self):
        return float(lib().dlz4_last_kernel_ms(self._h))

    def kernel_probe(self, enable=True, read=False):
        """Measurement aid (dlz4_kernel_probe): time the match finder and the encoder of fresh-block batches separately.
        read=True returns (finder_ms, encoder_ms) of the most recent probed batch."""
        a, b = C.c_float(0), C.c_float(0)
        self.check(lib().dlz4_kernel_probe(self._h, int(bool(enable)), C.byref(a) if read else None, C.byref(b) if read else None))
        return (a.value, b.value) if read else None

    @property
    def segment_stats(self):
        """(segments, re-run segments, rounds) of the most recent segment-parallel frame compression."""
        a, b, c = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
        lib().dlz4_segment_stats(self._h, C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value


_default = {}


def default_context(device=None):
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _default:
        _default[device] = Context(device)
    return _default[device]


# ---------------------------------------------------------------------------------------------- helpers
def compress_bound(n):
    return int(lib().dlz4_compress_bound(int(n)))


def frame_bound(n):
    return int(lib().dlz4_frame_bound(int(n)))


def host_register(array):
    """Page-locks a caller-owned numpy buffer (dlz4_host_register); True when the driver accepted it."""
    return lib().dlz4_host_register(_ptr(array), int(array.nbytes)) == 0


def host_unregister(array):
    return lib().dlz4_host_unregister(_ptr(array)) == 0


def shard_range(nblocks, world, rank):
    """Contiguous block range of `rank` (SURVEY 8e): returns (first, count)."""
    first, count = C.c_uint64(), C.c_uint64()
    lib().dlz4_shard_range(int(nblocks), int(world), int(rank), C.byref(first), C.byref(count))
    return int(first.value), int(count.value)


# ---------------------------------------------------------------------------------------------- raw block layer
def compressBlock(src, output, srcStart, srcLen, hashTable, outputOffset=0, ctx=None):
    """LZ4.compressRaw.  `output` (uint8 ndarray) and `hashTable` (int32[16384] ndarray) are written in place;
    returns the number of bytes written (which, as in the JS, may exceed what fitted into `output`)."""
    ctx = ctx or default_context()
    src = ensureBuffer(src)
    if not (isinstance(hashTable, np.ndarray) and hashTable.dtype == np.int32 and hashTable.size == 16384):
        raise TypeError("hashTable must be an int32 ndarray of 16384 entries")
    if not (isinstance(output, np.ndarray) and output.dtype == np.uint8):
        raise TypeError("output must be a uint8 ndarray")
    written = C.c_int32()
    st = lib().dlz4_compress_block(ctx.handle, _ptr(src), src.size, int(srcStart), int(srcLen), hashTable.ctypes.data,
                                   _ptr(output), output.size, int(outputOffset), C.byref(written))
    ctx.check(st)
    return int(written.value)


def decompressBlock(input, inputOffset, inputSize, output, outputOffset, dictionary=None, ctx=None):
    """LZ4.decompressRaw.  Writes into `output` (uint8 ndarray) at outputOffset; returns bytes written; raises LZ4Error
    with the reference's messages."""
    ctx = ctx or default_context()
    inp = ensureBuffer(input)
    if not (isinstance(output, np.ndarray) and output.dtype == np.uint8):
        raise TypeError("output must be a uint8 ndarray")
    d = ensureBuffer(dictionary) if dictionary is not None else None
    written = C.c_int64()
    st = lib().dlz4_decompress_block(ctx.handle, _ptr(inp), inp.size, int(inputOffset), int(inputSize), _ptr(output),
                                     output.size, int(outputOffset), _ptr(d), d.size if d is not None else 0,
                                     C.byref(written))
    ctx.check(st)
    return int(written.value)


def compress_blocks(src, off, length, prefix=None, warm=WARM_NONE, init_table=None, ctx=None, packed=False):
    """Batched compressBlock over independent blocks.  Returns (dst, dst_off, comp_len).
    packed=True: blocks are written back to back (dst_off = running sum of comp_len) through the chunked PCIe pipeline."""
    ctx = ctx or default_context()
    src = ensureBuffer(src)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    length = np.ascontiguousarray(length, dtype=np.uint32)
    n = len(off)
    if packed:
        dst = np.empty(int((length.astype(np.uint64) + length.astype(np.uint64) // 255 + 16).sum()), dtype=np.uint8)
        comp = np.zeros(n, dtype=np.uint32)
        p = ensureBuffer(prefix) if prefix is not None else None
        t = np.ascontiguousarray(init_table, dtype=np.int32) if init_table is not None else None
        st = lib().dlz4_compress_blocks(ctx.handle, _ptr(src), src.size, _ptr(off), _ptr(length), n, _ptr(p),
                                        p.size if p is not None else 0, int(warm), _ptr(t), _ptr(dst), dst.size, None, _ptr(comp))
        ctx.check(st)
        dst_off = np.zeros(n, dtype=np.uint64)
        if n:
            dst_off[1:] = np.cumsum(comp.astype(np.uint64))[:-1]
        return dst[:int(comp.astype(np.uint64).sum())], dst_off, comp
    bounds = (length.astype(np.uint64) + length.astype(np.uint64) // 255 + 16 + 15) & ~np.uint64(15)
    dst_off = np.zeros(n, dtype=np.uint64)
    if n:
        dst_off[1:] = np.cumsum(bounds)[:-1]
    dst = np.zeros(int(bounds.sum()), dtype=np.uint8)
    comp = np.zeros(n, dtype=np.uint32)
    p = ensureBuffer(prefix) if prefix is not None else None
    t = np.ascontiguousarray(init_table, dtype=np.int32) if init_table is not None else None
    st = lib().dlz4_compress_blocks(ctx.handle, _ptr(src), src.size, _ptr(off), _ptr(length), n, _ptr(p),
                                    p.size if p is not None else 0, int(warm), _ptr(t), _ptr(dst), dst.size, _ptr(dst_off),
                                    _ptr(comp))
    ctx.check(st)
    return dst, dst_off, comp


def decompress_blocks(src, off, length, dst_off, dst_cap, dictionary=None, hist_mode=HIST_RAW, ctx=None, check=True):
    """Batched decompressBlock.  Returns (dst, out_len, status)."""
    ctx = ctx or default_context()
    src = ensureBuffer(src)
    off = np.ascontiguousarray(off, dtype=np.uint64) if off is not None else None      # None: packed input
    length = np.ascontiguousarray(length, dtype=np.uint32)
    dst_off = np.ascontiguousarray(dst_off, dtype=np.uint64)
    dst_cap = np.ascontiguousarray(dst_cap, dtype=np.uint32)
    n = len(length)
    total = int((dst_off + dst_cap).max()) if n else 0
    dst = np.zeros(total, dtype=np.uint8)
    out_len = np.zeros(n, dtype=np.uint32)
    status = np.zeros(n, dtype=np.uint8)
    d = ensureBuffer(dictionary) if dictionary is not None else None
    st = lib().dlz4_decompress_blocks(ctx.handle, _ptr(src), src.size, _ptr(off), _ptr(length), n, _ptr(dst), dst.size,
                                      _ptr(dst_off), _ptr(dst_cap), _ptr(d), d.size if d is not None else 0, int(hist_mode),
                                      _ptr(out_len), _ptr(status))
    if check or st == E_CUDA or st >= 20:
        ctx.check(st)
    return dst, out_len, status


# ---------------------------------------------------------------------------------------------- xxHash32
def xxHash32(input, seed=0, ctx=None):
    ctx = ctx or default_context()
    a = ensureBuffer(input)
    out = C.c_uint32()
    ctx.check(lib().dlz4_xxh32(ctx.handle, _ptr(a), a.size, int(seed) & 0xFFFFFFFF, C.byref(out)))
    return int(out.value)


def xxh32_batch(base, off, length, seed=0, ctx=None):
    ctx = ctx or default_context()
    base = ensureBuffer(base)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    length = np.ascontiguousarray(length, dtype=np.uint32)
    out = np.zeros(len(off), dtype=np.uint32)
    ctx.check(lib().dlz4_xxh32_batch(ctx.handle, _ptr(base), base.size, _ptr(off), _ptr(length), len(off),
                                     int(seed) & 0xFFFFFFFF, _ptr(out)))
    return out


# ---------------------------------------------------------------------------------------------- frame layer
def compressBuffer(input, dictionary=None, maxBlockSize=4194304, blockIndependence=False, contentChecksum=False,
                   addContentSize=True, outputBuffer=None, blockChecksum=False, ctx=None):
    """LZ4.compress.  Returns the frame as bytes, or -- when outputBuffer (uint8 ndarray) is given -- a view of it,
    exactly like the reference's `output.subarray(0, outPos)` (bufferCompress.js:255)."""
    ctx = ctx or default_context()
    raw = ensureBuffer(input)
    d = ensureBuffer(dictionary) if dictionary is not None and len(dictionary) > 0 else None
    opts = FrameOpts(int(maxBlockSize or 0) & 0xFFFFFFFF if (maxBlockSize or 0) < 2 ** 32 else 0xFFFFFFFF,
                     int(bool(blockIndependence)), int(bool(contentChecksum)), int(bool(addContentSize)),
                     int(bool(blockChecksum)))
    if outputBuffer is None:
        out = np.empty(max(19 + raw.size + raw.size // 255 + 64 + 8, frame_bound(raw.size)), dtype=np.uint8)
    else:
        out = outputBuffer
    n = C.c_uint64()
    st = lib().dlz4_frame_compress(ctx.handle, _ptr(raw), raw.size, _ptr(d), d.size if d is not None else 0,
                                   C.byref(opts), _ptr(out), out.size, C.byref(n))
    ctx.check(st)
    used = min(int(n.value), out.size)
    return out[:used] if outputBuffer is not None else out[:used].tobytes()


def frame_info(frame):
    f = ensureBuffer(frame)
    info = FrameInfo()
    st = lib().dlz4_frame_info(_ptr(f), f.size, C.byref(info))
    if st:
        extra = " %d" % info.version if st == E_BAD_VERSION else ""
        raise LZ4Error(st, lib().dlz4_strerror(st).decode() + extra)
    return info


def decompressBuffer(input, dictionary=None, verifyChecksum=True, verifyBlockChecksums=False, ctx=None):
    """LZ4.decompress.  Returns bytes."""
    ctx = ctx or default_context()
    f = ensureBuffer(input)
    info = frame_info(f)
    d = ensureBuffer(dictionary) if dictionary is not None and len(dictionary) > 0 else None
    out = np.empty(int(info.max_decoded) + 16, dtype=np.uint8)
    n = C.c_uint64()
    flags = (1 if verifyChecksum else 0) | (2 if verifyBlockChecksums else 0)
    st = lib().dlz4_frame_decompress(ctx.handle, _ptr(f), f.size, _ptr(d), d.size if d is not None else 0, flags,
                                     _ptr(out), int(info.max_decoded), C.byref(n))
    ctx.check(st)
    return out[:int(n.value)].tobytes()


def decompressFrames(input, dictionary=None, verifyChecksum=True, verifyBlockChecksums=False, ctx=None):
    """Every LZ4 frame of a buffer of concatenated frames, skippable frames skipped (SURVEY 8 f3; the reference's
    decompressBuffer stops at the first EndMark, its stream decoder loops: src/shared/lz4Decode.js:262-266).
    Returns (bytes, number of frames)."""
    ctx = ctx or default_context()
    f = ensureBuffer(input)
    total, count = C.c_uint64(0), C.c_uint32(0)
    st = lib().dlz4_frames_info(_ptr(f), f.size, C.byref(total), C.byref(count))
    ctx.check(st)
    d = ensureBuffer(dictionary) if dictionary is not None and len(dictionary) > 0 else None
    out = np.empty(int(total.value) + 16, dtype=np.uint8)
    n = C.c_uint64()
    flags = (1 if verifyChecksum else 0) | (2 if verifyBlockChecksums else 0)
    st = lib().dlz4_frames_decompress(ctx.handle, _ptr(f), f.size, _ptr(d), d.size if d is not None else 0, flags,
                                      _ptr(out), int(total.value), C.byref(n), C.byref(count))
    ctx.check(st)
    return out[:int(n.value)].tobytes(), int(count.value)


def frame_opts(maxBlockSize=4194304, blockIndependence=False, contentChecksum=False, addContentSize=True, blockChecksum=False):
    """The dlz4_frame_opts of compressBuffer's arguments."""
    return FrameOpts(int(maxBlockSize or 0) & 0xFFFFFFFF if (maxBlockSize or 0) < 2 ** 32 else 0xFFFFFFFF,
                     int(bool(blockIndependence)), int(bool(contentChecksum)), int(bool(addContentSize)), int(bool(blockChecksum)))


def _concat(items):
    """Packs a list of byte-likes into one uint8 array: (array, offsets u64, lengths)."""
    arrs = [ensureBuffer(x) for x in items]
    lens = np.array([a.size for a in arrs], dtype=np.uint64)
    off = np.zeros(len(arrs), dtype=np.uint64)
    if len(arrs) > 1:
        off[1:] = np.cumsum(lens)[:-1]
    buf = np.concatenate(arrs) if arrs else np.zeros(0, dtype=np.uint8)
    return np.ascontiguousarray(buf, dtype=np.uint8), off, lens


def _frame_error(status, frame):
    """LZ4Error of a frame's status, with the version read from its FLG byte for "Unsupported Version N"."""
    extra = ""
    if status == E_BAD_VERSION:
        f = ensureBuffer(frame)
        extra = " %d" % ((int(f[4]) & 0xC0) >> 6 if f.size >= 5 else 0)
    return LZ4Error(status, lib().dlz4_strerror(status).decode() + extra)


def compressBuffers(inputs, dictionary=None, maxBlockSize=4194304, blockIndependence=False, contentChecksum=False,
                    addContentSize=True, blockChecksum=False, ctx=None):
    """compressBuffer over many inputs in one GPU pass (dlz4_frames_compress_batch): one frame per input, each byte-identical
    to compressBuffer(input, dictionary, ...) with the same options.  Returns a list of bytes."""
    ctx = ctx or default_context()
    src, off, lens = _concat(inputs)
    n = len(lens)
    if n == 0:
        return []
    d = ensureBuffer(dictionary) if dictionary is not None and len(dictionary) > 0 else None
    opts = frame_opts(maxBlockSize, blockIndependence, contentChecksum, addContentSize, blockChecksum)
    lens32 = lens.astype(np.uint32)
    if (lens >= 0x7FFF0000).any():
        ctx.check(21)
    cap = int((19 + lens + (lens // 65536 + 1) * 8 + 8 + 64).sum())
    dst = np.empty(cap, dtype=np.uint8)
    frame_off = np.zeros(n + 1, dtype=np.uint64)
    st = lib().dlz4_frames_compress_batch(ctx.handle, _ptr(src), src.size, _ptr(off), _ptr(lens32), n, _ptr(d),
                                          d.size if d is not None else 0, C.byref(opts), _ptr(dst), cap, _ptr(frame_off))
    ctx.check(st)
    fo = frame_off.tolist()
    mv = dst.tobytes()
    return [mv[fo[i]:fo[i + 1]] for i in range(n)]


def decompressBuffers(frames, dictionary=None, verifyChecksum=True, verifyBlockChecksums=False, errors="raise", ctx=None):
    """decompressBuffer over many frames in one GPU pass (dlz4_frames_batch_info + dlz4_frames_decompress_batch).  Entry i is
    what decompressBuffer(frames[i], ...) returns.  errors="raise": the first failing frame's LZ4Error is raised;
    errors="return": a failing frame's entry is its LZ4Error."""
    if errors not in ("raise", "return"):
        raise ValueError('errors must be "raise" or "return"')
    ctx = ctx or default_context()
    src, off, lens = _concat(frames)
    n = len(lens)
    if n == 0:
        return []
    L = lib()
    max_dec = np.zeros(n, dtype=np.uint64)
    info_st = np.zeros(n, dtype=np.uint8)
    ctx.check(L.dlz4_frames_batch_info(ctx.handle, _ptr(src), src.size, _ptr(off), _ptr(lens), n, _ptr(max_dec), _ptr(info_st)))
    dst_cap = max_dec
    dst_off = np.zeros(n, dtype=np.uint64)
    if n > 1:
        dst_off[1:] = np.cumsum(dst_cap)[:-1]
    total = int(dst_cap.sum())
    dst = np.empty(total + 16, dtype=np.uint8)
    out_len = np.zeros(n, dtype=np.uint64)
    status = np.zeros(n, dtype=np.uint8)
    d = ensureBuffer(dictionary) if dictionary is not None and len(dictionary) > 0 else None
    flags = (1 if verifyChecksum else 0) | (2 if verifyBlockChecksums else 0)
    st = L.dlz4_frames_decompress_batch(ctx.handle, _ptr(src), src.size, _ptr(off), _ptr(lens), n, _ptr(d),
                                        d.size if d is not None else 0, flags, _ptr(dst), dst.size, _ptr(dst_off), _ptr(dst_cap),
                                        _ptr(out_len), _ptr(status))
    if st == E_CUDA or st >= 20:
        ctx.check(st)
    out = []
    mv = dst.tobytes()
    for i in range(n):
        s = int(info_st[i]) or int(status[i])               # decompressBuffer raises frame_info's error first
        if s:
            e = _frame_error(s, frames[i])
            if errors == "raise":
                raise e
            out.append(e)
        else:
            o = int(dst_off[i])
            out.append(mv[o:o + int(out_len[i])])
    return out


class XXHash32(object):
    """The reference's stateful hasher (src/xxhash32/xxhash32Stateful.js): update(bytes) ... digest()."""

    def __init__(self, seed=0, ctx=None):
        self._ctx = ctx or default_context()
        self._s = Xxh32State()
        lib().dlz4_xxh32_reset(C.byref(self._s), seed & 0xFFFFFFFF)

    def update(self, data):
        b = ensureBuffer(data)
        if b.size:
            self._ctx.check(lib().dlz4_xxh32_update(self._ctx.handle, C.byref(self._s), _ptr(b), b.size))
        return self

    def update_resident(self, which):
        """Continues over bytes the last frame / stream call left on the device (0: its input, 1: its decoded output) instead
        of uploading them again; False when the state holds a partial stripe (the caller then updates from host bytes)."""
        if self._s.memsize:
            return False
        self._ctx.check(lib().dlz4_xxh32_update_resident(self._ctx.handle, C.byref(self._s), int(which)))
        return True

    def digest(self):
        return int(lib().dlz4_xxh32_digest(C.byref(self._s)))


def chain_compress(work, start, total, block_size, table, ctx=None):
    """Every block of work[start, start+total) as one linked chain, `table` (int32[16384]) carried in and out
    (LZ4Encoder._flushBlock over all full blocks of an add(), lz4Encode.js:215-298).  Returns a list of per-block bytes."""
    ctx = ctx or default_context()
    work = ensureBuffer(work)
    n = (total + block_size - 1) // block_size
    if n == 0:
        return []
    stride = compress_bound(block_size)
    dst = np.empty(n * stride, dtype=np.uint8)
    clen = np.zeros(n, dtype=np.uint32)
    st = lib().dlz4_chain_compress(ctx.handle, _ptr(work), work.size, int(start), int(total), int(block_size), _ptr(table),
                                   _ptr(dst), stride, _ptr(clen))
    ctx.check(st)
    return [dst[k * stride:k * stride + int(clen[k])] for k in range(n)]


class _LZ4(object):
    """The reference's facade object (src/lz4.js:27-66): block / buffer members, the stream classes and the worker offload."""
    compressRaw = staticmethod(compressBlock)
    decompressRaw = staticmethod(decompressBlock)
    compress = staticmethod(compressBuffer)
    decompress = staticmethod(decompressBuffer)
    xxHash32 = staticmethod(xxHash32)

    @staticmethod
    def compressWorker(data, options=None):                    # src/lz4.js:54
        from .worker import LZ4Worker
        return LZ4Worker.compress(data, options)

    @staticmethod
    def decompressWorker(data, options=None):                  # src/lz4.js:55
        from .worker import LZ4Worker
        return LZ4Worker.decompress(data, options)

    @staticmethod
    def compressWorkerStream(readable, writable, options=None):    # src/lz4.js:58 (LZ4Worker.compressStream)
        from .worker import LZ4Worker
        return LZ4Worker.compressStream(readable, writable, options)

    @staticmethod
    def decompressWorkerStream(readable, writable, options=None):  # src/lz4.js:59
        from .worker import LZ4Worker
        return LZ4Worker.decompressStream(readable, writable, options)


LZ4 = _LZ4()
