"""Concatenated frames in device memory (compress_tensor_frames / decompress_tensor_frames) against the routes a user has
without them, with a check that every route gives the same bytes.
  1. 4.5 GiB MIXED with content checksums, in independent 64 KiB blocks and in the default linked 4 MiB frame (5 frames:
     four of 1 GiB, one of 0.5 GiB): the frame-sequence calls; a Python loop of compress_tensor / decompress_tensor over the
     same spans; compress_sharded / decompress_sharded with one rank on page-locked host buffers.  Also timed on their own:
     one k_xxh32_stream chain over a 1 GiB span, and frames_info_dev (the one-thread k_fs_walk of the sequence + one sync).
  2. 100 000 concatenated 4 KiB JSON frames (compressBuffers): decompress_tensor_frames against api.decompressFrames on host
     memory and against frames_decompress_batch_dev with the frame offsets already known.
  3. The route threshold (DLZ4_FRAMES_WARP_MAX_KIB, default 4 MiB of max_decoded): 256 MiB of log text as linked 64 KiB-block
     frames of 2 MiB (below) and of 16 MiB (above), decoded by the default context and by contexts that force each route.
Rates are GB/s of uncompressed bytes, best of `reps` runs.  The first line names the card, its power limit and SM clocks,
read in the same run.
Usage: python divortio-lz4_b200/tools/frames_dev_bench.py [reps] [out.txt]   (default 3; the report also goes to out.txt)"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import divortio_lz4_b200 as dl  # noqa: E402
from divortio_lz4_b200 import corpus, device as dev, sharded  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
out_path = sys.argv[2] if len(sys.argv) > 2 else None
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True)
say("card (name, power limit, SM clock, max SM clock): %s" % q.stdout.strip())
ctx = dl.default_context(0)
cuda = torch.device("cuda", 0)


def best(fn):
    t_best, r = 1e9, None
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        t_best = min(t_best, time.perf_counter() - t)
    return t_best, r


def pinned(n):
    return torch.empty(max(n, 1), dtype=torch.uint8, pin_memory=True).numpy()[:n]


def new_ctx(**env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return dl.Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


# ---------------------------------------------------------------------------------------------------------------- 1.
n = (9 << 30) // 2
data = corpus.mixed(1, n)
h_in = pinned(n)
h_in[:] = data
t_in = torch.from_numpy(data).to(cuda)
del data
spans = sharded.frame_spans(n)
gb = n / 1e9
x = torch.empty(1, dtype=torch.int32, device=cuda)
t_chain, _ = best(lambda: dev.xxh32_stream_dev(ctx, t_in[:1 << 30], x))
say("\n1. 4.5 GiB MIXED, contentChecksum=True, %d frames; one k_xxh32_stream chain over 1 GiB: %.3f s" % (len(spans), t_chain))
say("%-34s %12s %12s %12s %12s %12s %12s %10s" % ("options", "c frames", "c loop", "c sharded", "d frames", "d loop",
                                                  "d sharded", "walk"))
for name, kw, bs in (("independent 64 KiB blocks", dict(maxBlockSize=65536, blockIndependence=True), 65536),
                     ("default frame (linked 4 MiB)", dict(), 4194304)):
    t_cf, f = best(lambda: dev.compress_tensor_frames(t_in, contentChecksum=True, **kw))
    t_cl, parts = best(lambda: [dev.compress_tensor(t_in[lo:hi], contentChecksum=True, **kw) for lo, hi in spans])
    assert torch.equal(f, torch.cat(parts)), name
    foff = np.concatenate([[0], np.cumsum([p.numel() for p in parts])])
    del parts
    h_out = pinned(f.numel() + (1 << 20))
    back = pinned(n + 64)
    be = sharded.GpuBackend(ctx)
    if kw.get("blockIndependence"):
        t_cs, total = best(lambda: sharded.compress_sharded(h_in, h_out, bs, True, True, False, comm=sharded.LocalComm(), backend=be))
        assert total == f.numel() and np.array_equal(h_out[:total], f.cpu().numpy()), name
    else:
        t_cs = float("nan")                                  # compress_sharded writes independent blocks only
        h_out[:f.numel()] = f.cpu().numpy()
        total = f.numel()
    t_ds, got = best(lambda: sharded.decompress_sharded(h_out[:total], back, True, False, comm=sharded.LocalComm(), backend=be))
    assert got == n and np.array_equal(back[:n], h_in), name
    del back, h_out
    t_df, (out, k) = best(lambda: dev.decompress_tensor_frames(f))
    assert k == len(spans) and torch.equal(out, t_in), name
    del out
    t_dl, outs = best(lambda: [dev.decompress_tensor(f[foff[i]:foff[i + 1]]) for i in range(len(spans))])
    assert torch.equal(torch.cat(outs), t_in), name
    del outs
    t_walk, _ = best(lambda: dev.frames_info_dev(ctx, f))
    say("%-34s %12.2f %12.2f %12.2f %12.2f %12.2f %12.2f %8.3fms" % (name, gb / t_cf, gb / t_cl, gb / t_cs, gb / t_df, gb / t_dl,
                                                                      gb / t_ds, t_walk * 1e3))
    del f
    torch.cuda.empty_cache()
say("c/d frames: compress_tensor_frames / decompress_tensor_frames;  c/d loop: compress_tensor / decompress_tensor per span;  "
    "c/d sharded: compress_sharded / decompress_sharded, one rank, page-locked host buffers (GB/s);  walk: frames_info_dev")
del t_in, h_in
torch.cuda.empty_cache()

# ---------------------------------------------------------------------------------------------------------------- 2.
blob = corpus.jsonmsgs(2, 0, 100000)
msgs = [blob[i * 4096:(i + 1) * 4096].tobytes() for i in range(100000)]
frames = dl.compressBuffers(msgs)
host = np.frombuffer(b"".join(frames), dtype=np.uint8)
plain = b"".join(msgs)
gb = len(plain) / 1e9
f = torch.from_numpy(host.copy()).to(cuda)
t_df, (out, k) = best(lambda: dev.decompress_tensor_frames(f))
assert k == 100000 and out.cpu().numpy().tobytes() == plain
t_dh, (got, k) = best(lambda: dl.decompressFrames(host))
assert k == 100000 and got == plain
lens = np.array([len(x) for x in frames], dtype=np.int64)
foff = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)[:-1]])).to(cuda)
flen = torch.from_numpy(lens).to(cuda)
caps = torch.full((100000,), 4096, dtype=torch.int64, device=cuda)
doff = torch.arange(100000, dtype=torch.int64, device=cuda) * 4096
dst = torch.empty(100000 * 4096, dtype=torch.uint8, device=cuda)
olen = torch.empty(100000, dtype=torch.int64, device=cuda)
stat = torch.empty(100000, dtype=torch.uint8, device=cuda)
t_db, _ = best(lambda: dev.frames_decompress_batch_dev(ctx, f, foff, flen, dst, doff, caps, olen, stat))
assert not stat.any() and dst.cpu().numpy().tobytes() == plain
say("\n2. 100 000 concatenated 4 KiB JSON frames (%.1f MB): decompress_tensor_frames %.2f GB/s (%.2f ms);  decompressFrames "
    "(host memory) %.2f GB/s;  frames_decompress_batch_dev, offsets known: %.2f GB/s" % (len(plain) / 1e6, gb / t_df, t_df * 1e3,
                                                                                        gb / t_dh, gb / t_db))
del f, out, dst

# ---------------------------------------------------------------------------------------------------------------- 3.
say("\n3. route threshold: 256 MiB log text, linked 64 KiB-block frames; decompress_tensor_frames GB/s")
say("%-28s %12s %12s %12s" % ("frame size", "default", "all warp", "all alone"))
c_warp = new_ctx(DLZ4_FRAMES_WARP_MAX_KIB=str(1 << 40))
c_alone = new_ctx(DLZ4_FRAMES_WARP_MAX_KIB="0")
log = torch.from_numpy(corpus.log(3, 256 << 20)).to(cuda)
for size in (2 << 20, 16 << 20):
    f = dev.compress_tensor_frames(log, maxBlockSize=65536, frame_max=size)
    row = []
    for c in (ctx, c_warp, c_alone):
        t, (out, k) = best(lambda: dev.decompress_tensor_frames(f, ctx=c))
        assert torch.equal(out, log)
        row.append(log.numel() / 1e9 / t)
    say("%-28s %12.2f %12.2f %12.2f" % ("%d KiB (%d frames)" % (size >> 10, k), *row))
if out_path:
    with open(out_path, "w") as fh:
        fh.write("\n".join(lines) + "\n")
