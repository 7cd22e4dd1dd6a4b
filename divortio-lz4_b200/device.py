"""Device-resident entry points: torch CUDA tensors in, torch CUDA tensors out, no host copies.

torch is plumbing here (device memory + the current stream); the work is done by the _dev functions of the C ABI.
"""
import ctypes as C

import torch

from . import api, sharded


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None and t.numel() else None


def _stream(device=None):
    """Current torch stream (of `device`, default the current device) as the ABI's opaque handle.  torch's default stream has
    handle 0, which the ABI reads as "use the context's own stream", so it is passed as cudaStreamLegacy (0x1) instead."""
    h = torch.cuda.current_stream(device).cuda_stream
    return C.c_void_p(h if h else 1)


def uniform_blocks(total, block, device, dst_stride=None):
    """Block table of a contiguous buffer: (off u64, len u32, nblocks[, dst_off u64])."""
    n = (total + block - 1) // block
    idx = torch.arange(n, device=device, dtype=torch.int64)
    off = idx * block
    length = torch.clamp(total - off, max=block).to(torch.int32)
    if dst_stride is None:
        return off, length, n
    return off, length, n, idx * dst_stride


def compress_blocks_dev(ctx, src, src_off, src_len, max_block_len, dst, dst_off, comp_len, prefix=None, warm=api.WARM_NONE,
                        init_table=None):
    """dlz4_compress_blocks_dev on the current torch stream.  All arguments are CUDA tensors
    (src/dst/prefix uint8, *_off int64, *_len int32, init_table int32[16384])."""
    st = api.lib().dlz4_compress_blocks_dev(ctx.handle, _p(src), _p(src_off), _p(src_len), src_off.numel(), int(max_block_len),
                                            _p(prefix), prefix.numel() if prefix is not None else 0, int(warm), _p(init_table),
                                            _p(dst), _p(dst_off), _p(comp_len), _stream())
    ctx.check(st)


def decompress_blocks_dev(ctx, src, src_off, src_len, dst, dst_off, dst_cap, out_len, status, dictionary=None,
                          hist_mode=api.HIST_RAW):
    st = api.lib().dlz4_decompress_blocks_dev(ctx.handle, _p(src), _p(src_off), _p(src_len), src_off.numel(), _p(dst), _p(dst_off),
                                              _p(dst_cap), _p(dictionary), dictionary.numel() if dictionary is not None else 0,
                                              int(hist_mode), _p(out_len), _p(status), _stream())
    ctx.check(st)


def xxh32_batch_dev(ctx, base, off, length, out, seed=0):
    ctx.check(api.lib().dlz4_xxh32_batch_dev(ctx.handle, _p(base), _p(off), _p(length), off.numel(), seed, _p(out), _stream()))


def xxh32_stream_dev(ctx, data, out, seed=0):
    ctx.check(api.lib().dlz4_xxh32_stream_dev(ctx.handle, _p(data), data.numel(), seed, _p(out), _stream()))


def frame_pack_dev(ctx, src, src_off, src_len, comp, comp_off, comp_len, block_checksum, segment, block_pos):
    ctx.check(api.lib().dlz4_frame_pack_dev(ctx.handle, _p(src), _p(src_off), _p(src_len), _p(comp), _p(comp_off), _p(comp_len),
                                            src_off.numel(), int(block_checksum), _p(segment), _p(block_pos), _stream()))


def frames_compress_batch_dev(ctx, src, src_off, src_len, max_len, dst, frame_off, opts, dictionary=None):
    """dlz4_frames_compress_batch_dev on the current torch stream.  src/dst/dictionary uint8, src_off int64, src_len int32,
    frame_off int64[nframes + 1] (CUDA tensors); opts an api.FrameOpts (api.frame_opts(...))."""
    ctx.check(api.lib().dlz4_frames_compress_batch_dev(ctx.handle, _p(src), _p(src_off), _p(src_len), src_off.numel(), int(max_len),
                                                       _p(dictionary), dictionary.numel() if dictionary is not None else 0,
                                                       C.byref(opts), _p(dst), dst.numel(), _p(frame_off), _stream()))


def frames_batch_info_dev(ctx, src, frame_off, frame_len, max_decoded, status):
    """dlz4_frames_batch_info_dev: max_decoded int64, status uint8 (CUDA tensors, one entry per frame)."""
    ctx.check(api.lib().dlz4_frames_batch_info_dev(ctx.handle, _p(src), _p(frame_off), _p(frame_len), frame_off.numel(), _p(max_decoded),
                                                   _p(status), _stream()))


def frames_decompress_batch_dev(ctx, src, frame_off, frame_len, dst, dst_off, dst_cap, out_len, status, dictionary=None, flags=1):
    """dlz4_frames_decompress_batch_dev on the current torch stream; per-frame statuses land in `status` (uint8)."""
    ctx.check(api.lib().dlz4_frames_decompress_batch_dev(ctx.handle, _p(src), _p(frame_off), _p(frame_len), frame_off.numel(),
                                                         _p(dictionary), dictionary.numel() if dictionary is not None else 0,
                                                         int(flags), _p(dst), _p(dst_off), _p(dst_cap), _p(out_len), _p(status),
                                                         _stream()))


# ---------------------------------------------------------------------------------------------- single frames in device memory
def frame_compress_dev(ctx, src, dst, opts, dictionary=None):
    """dlz4_frame_compress_dev on the current torch stream.  src/dst/dictionary are uint8 CUDA tensors (any byte offset), dst
    at least api.frame_bound(src.numel()) bytes; opts an api.FrameOpts (api.frame_opts(...)).  Returns the frame's length."""
    n = C.c_uint64(0)
    ctx.check(api.lib().dlz4_frame_compress_dev(ctx.handle, _p(src), src.numel(), _p(dictionary),
                                                dictionary.numel() if dictionary is not None else 0, C.byref(opts), _p(dst), dst.numel(),
                                                C.byref(n), _stream(src.device)))
    return int(n.value)


def frame_info_dev(ctx, frame):
    """dlz4_frame_info_dev on the current torch stream: the api.FrameInfo of the frame in a uint8 CUDA tensor.  Raises
    api.LZ4Error with the reference's text, as api.frame_info does."""
    info = api.FrameInfo()
    st = api.lib().dlz4_frame_info_dev(ctx.handle, _p(frame), frame.numel(), C.byref(info), _stream(frame.device))
    ctx.check(st, " %d" % info.version if st == api.E_BAD_VERSION else "")
    return info


def frame_decompress_dev(ctx, frame, dst, dictionary=None, flags=1):
    """dlz4_frame_decompress_dev on the current torch stream: decodes the frame in `frame` into `dst` (uint8 CUDA tensors, the
    capacity is dst.numel()).  flags: bit 0 content checksum, bit 1 block checksums, bit 2 header checksum.  Returns the
    decoded length."""
    n = C.c_uint64(0)
    ctx.check(api.lib().dlz4_frame_decompress_dev(ctx.handle, _p(frame), frame.numel(), _p(dictionary),
                                                  dictionary.numel() if dictionary is not None else 0, int(flags), _p(dst), dst.numel(),
                                                  C.byref(n), _stream(frame.device)))
    return int(n.value)


def _bytes_of(t, name, ctx):
    """A contiguous CUDA tensor viewed as uint8 bytes, on the context's device."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor" % name)
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    if ctx is not None and t.device.index != ctx.device:
        raise ValueError("%s is on %s, the context on cuda:%d" % (name, t.device, ctx.device))
    return t.reshape(-1).view(torch.uint8)


def _dictionary_on(dictionary, device, ctx):
    if dictionary is None:
        return None
    if isinstance(dictionary, torch.Tensor):
        d = _bytes_of(dictionary, "dictionary", ctx)
    else:
        d = torch.from_numpy(api.ensureBuffer(dictionary).copy()).to(device)
    return d if d.numel() else None


def compress_tensor(t, dictionary=None, maxBlockSize=4194304, blockIndependence=False, contentChecksum=False, addContentSize=True,
                    blockChecksum=False, ctx=None):
    """LZ4.compress of a CUDA tensor's bytes, on the GPU end to end: returns a uint8 CUDA tensor of exactly the frame's length,
    byte-identical to compressBuffer(t's bytes, ...).  t: any contiguous CUDA tensor; dictionary: a CUDA tensor or bytes-like.
    Runs on the current torch stream and returns when the frame is complete."""
    src = _bytes_of(t, "t", ctx)
    ctx = ctx or api.default_context(src.device.index)
    d = _dictionary_on(dictionary, src.device, ctx)
    dst = torch.empty(api.frame_bound(src.numel()), dtype=torch.uint8, device=src.device)
    n = frame_compress_dev(ctx, src, dst, api.frame_opts(maxBlockSize, blockIndependence, contentChecksum, addContentSize, blockChecksum), d)
    return dst[:n]


def decompress_tensor(frame, dictionary=None, verifyChecksum=True, verifyBlockChecksums=False, ctx=None):
    """LZ4.decompress of a frame held in a CUDA tensor, on the GPU end to end: returns the decoded bytes as a uint8 CUDA tensor
    (sized with frame_info_dev).  Raises api.LZ4Error with the reference's text, as decompressBuffer does."""
    f = _bytes_of(frame, "frame", ctx)
    ctx = ctx or api.default_context(f.device.index)
    d = _dictionary_on(dictionary, f.device, ctx)
    info = frame_info_dev(ctx, f)
    out = torch.empty(int(info.max_decoded), dtype=torch.uint8, device=f.device)
    n = frame_decompress_dev(ctx, f, out, d, (1 if verifyChecksum else 0) | (2 if verifyBlockChecksums else 0))
    return out[:n]


# ---------------------------------------------------------------------------------------- concatenated frames in device memory
def frames_compress_dev(ctx, src, frame_bytes, dst, opts, dictionary=None):
    """dlz4_frames_compress_dev on the current torch stream: src cut into spans of frame_bytes, one frame each, back to back in
    dst (uint8 CUDA tensors, dst at least the sum of api.frame_bound over the spans).  Returns (length, frame_off list)."""
    n, k = C.c_uint64(0), C.c_uint32(0)
    spans = max(1, -(-src.numel() // int(frame_bytes))) if frame_bytes else 1
    off = (C.c_uint64 * (spans + 1))()
    ctx.check(api.lib().dlz4_frames_compress_dev(ctx.handle, _p(src), src.numel(), int(frame_bytes), _p(dictionary),
                                                 dictionary.numel() if dictionary is not None else 0, C.byref(opts), _p(dst),
                                                 dst.numel(), off, C.byref(n), C.byref(k), _stream(src.device)))
    return int(n.value), [int(x) for x in off[:k.value + 1]]


def frames_info_dev(ctx, data):
    """dlz4_frames_info_dev on the current torch stream: (sum of max_decoded, LZ4 frames) of the concatenated frames in a uint8
    CUDA tensor.  Raises api.LZ4Error as api.decompressFrames does."""
    total, count = C.c_uint64(0), C.c_uint32(0)
    ctx.check(api.lib().dlz4_frames_info_dev(ctx.handle, _p(data), data.numel(), C.byref(total), C.byref(count), _stream(data.device)))
    return int(total.value), int(count.value)


def frames_decompress_dev(ctx, data, dst, dictionary=None, flags=1):
    """dlz4_frames_decompress_dev on the current torch stream: every LZ4 frame of `data` in order into `dst` (capacity
    dst.numel()), skippable frames skipped.  Returns (decoded length, frames)."""
    n, count = C.c_uint64(0), C.c_uint32(0)
    ctx.check(api.lib().dlz4_frames_decompress_dev(ctx.handle, _p(data), data.numel(), _p(dictionary),
                                                   dictionary.numel() if dictionary is not None else 0, int(flags), _p(dst), dst.numel(),
                                                   C.byref(n), C.byref(count), _stream(data.device)))
    return int(n.value), int(count.value)


def compress_tensor_frames(t, dictionary=None, maxBlockSize=4194304, blockIndependence=False, contentChecksum=False,
                           addContentSize=True, blockChecksum=False, frame_max=sharded.FRAME_MAX, ctx=None):
    """compress_tensor for a CUDA tensor of any size: frames cut by sharded.frame_spans (one frame up to frame_max bytes, else
    frames of sharded.FRAME_SPLIT bytes, or of frame_max bytes when the caller sets a limit), back to back in one uint8 CUDA
    tensor.  Up to frame_max bytes the result is compress_tensor's frame; the content checksums of several frames are computed
    side by side."""
    src = _bytes_of(t, "t", ctx)
    ctx = ctx or api.default_context(src.device.index)
    d = _dictionary_on(dictionary, src.device, ctx)
    spans = sharded.frame_spans(src.numel(), frame_max)
    step = max(1, spans[0][1] - spans[0][0])
    dst = torch.empty(sum(api.frame_bound(hi - lo) for lo, hi in spans), dtype=torch.uint8, device=src.device)
    n, _ = frames_compress_dev(ctx, src, step, dst,
                               api.frame_opts(maxBlockSize, blockIndependence, contentChecksum, addContentSize, blockChecksum), d)
    return dst[:n]


def decompress_tensor_frames(data, dictionary=None, verifyChecksum=True, verifyBlockChecksums=False, ctx=None):
    """api.decompressFrames of concatenated frames held in a CUDA tensor, on the GPU end to end: returns (uint8 CUDA tensor of
    the decoded bytes, number of LZ4 frames).  Raises api.LZ4Error with the reference's text."""
    f = _bytes_of(data, "data", ctx)
    ctx = ctx or api.default_context(f.device.index)
    d = _dictionary_on(dictionary, f.device, ctx)
    total, _ = frames_info_dev(ctx, f)
    out = torch.empty(total, dtype=torch.uint8, device=f.device)
    n, count = frames_decompress_dev(ctx, f, out, d, (1 if verifyChecksum else 0) | (2 if verifyBlockChecksums else 0))
    return out[:n], count
