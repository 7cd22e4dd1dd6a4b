"""Device-resident entry points: torch CUDA tensors in, torch CUDA tensors out, no host copies.

torch is plumbing here (device memory + the current stream); the work is done by the _dev functions of the C ABI.
"""
import ctypes as C

import torch

from . import api


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None and t.numel() else None


def _stream():
    """Current torch stream as the ABI's opaque handle.  torch's default stream has handle 0, which the ABI reads as
    "use the context's own stream", so it is passed as cudaStreamLegacy (0x1) instead."""
    h = torch.cuda.current_stream().cuda_stream
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
