"""Batched frames against the per-frame loop, configs[3] shape: 4 KiB JSON messages behind the 64 KiB dictionary, each message
its own LZ4 frame (the reference's LZ4.compress / LZ4.decompress once per message).  Prints, in one run:
  the card (name, power limit, SM clock);
  the per-frame compressBuffer / decompressBuffer loop on a sample (us per frame);
  compressBuffers / decompressBuffers host to host, and the _dev calls device-resident (GB/s of message bytes, messages/s);
  the raw-block calls on the same messages (dlz4_compress_blocks_dev / dlz4_decompress_blocks_dev, prefix + Jenkins table);
  a crossover sweep over frame size (64 KiB .. 64 MiB at the same total bytes): batch call against a loop of single-frame calls.
Usage: python divortio-lz4_b200/tools/frame_batch_bench.py [messages] [sample]   (defaults 1048576, 20000)"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import divortio_lz4_b200 as dl  # noqa: E402
from divortio_lz4_b200 import corpus, device as dev  # noqa: E402

count = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
sample = int(sys.argv[2]) if len(sys.argv) > 2 else 20000
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
print("card: %s" % q.stdout.strip(), flush=True)
ctx = dl.Context(0)
d = torch.device("cuda", 0)
raw = corpus.jsonmsgs(4, 0, count)
dic = corpus.json_dictionary(44).tobytes()
rawb = raw.tobytes()
msgs = [rawb[i * 4096:(i + 1) * 4096] for i in range(count)]
tot = count * 4096


def timed(fn, reps=3):
    best = 1e9
    r = None
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t)
    return best, r


for cc in (False, True):
    tag = "cc=%d" % cc
    # per-frame loop on a sample
    sm = msgs[:sample]
    tl, one = timed(lambda: [dl.compressBuffer(m, dic, 4194304, False, cc, ctx=ctx) for m in sm], 1)
    tdl, _ = timed(lambda: [dl.decompressBuffer(f, dic, True, ctx=ctx) for f in one], 1)
    print("%s per-frame loop (%d frames): compress %.1f us/frame, decompress %.1f us/frame" % (tag, sample, tl / sample * 1e6,
                                                                                                tdl / sample * 1e6), flush=True)
    # batch, host to host
    tc, frames = timed(lambda: dl.compressBuffers(msgs, dic, contentChecksum=cc, ctx=ctx))
    assert frames[:sample] == one
    td, back = timed(lambda: dl.decompressBuffers(frames, dic, ctx=ctx))
    assert back == msgs
    print("%s batch host-to-host (%d frames, Python packing included): compress %.2f GB/s (%.2f M msgs/s), decompress %.2f GB/s "
          "(%.2f M msgs/s)" % (tag, count, tot / tc / 1e9, count / tc / 1e6, tot / td / 1e9, count / td / 1e6), flush=True)
    # batch, device-resident
    src = torch.from_numpy(raw).to(d)
    off = torch.arange(count, dtype=torch.int64, device=d) * 4096
    ln = torch.full((count,), 4096, dtype=torch.int32, device=d)
    t_dic = torch.frombuffer(bytearray(dic), dtype=torch.uint8).to(d)
    cap = count * dl.frame_bound(4096)
    dst = torch.empty(cap, dtype=torch.uint8, device=d)
    fo = torch.zeros(count + 1, dtype=torch.int64, device=d)
    opts = dl.api.frame_opts(4194304, False, cc, True, False)
    tcd, _ = timed(lambda: dev.frames_compress_batch_dev(ctx, src, off, ln, 4096, dst, fo, opts, t_dic))
    flen = fo[1:] - fo[:-1]
    foff = fo[:-1].contiguous()
    out = torch.empty(tot + 64, dtype=torch.uint8, device=d)
    doff = off.clone()
    dcap = torch.full((count,), 4096, dtype=torch.int64, device=d)
    olen = torch.zeros(count, dtype=torch.int64, device=d)
    st = torch.zeros(count, dtype=torch.uint8, device=d)
    tdd, _ = timed(lambda: dev.frames_decompress_batch_dev(ctx, dst, foff, flen, out, doff, dcap, olen, st, t_dic, flags=1))
    assert int(st.max()) == 0 and torch.equal(out[:tot], src)
    print("%s batch device-resident: compress %.2f GB/s (%.2f M msgs/s), decompress %.2f GB/s (%.2f M msgs/s), frames %.1f MB"
          % (tag, tot / tcd / 1e9, count / tcd / 1e6, tot / tdd / 1e9, count / tdd / 1e6, int(fo[-1]) / 1e6), flush=True)

# raw blocks on the same messages (prefix + Jenkins-warmed table), device-resident
stride = (dl.compress_bound(4096) + 15) & ~15
comp = torch.empty(count * stride + 64, dtype=torch.uint8, device=d)
coff = torch.arange(count, dtype=torch.int64, device=d) * stride
clen = torch.zeros(count, dtype=torch.int32, device=d)
ln32 = torch.full((count,), 4096, dtype=torch.int32, device=d)
olen32 = torch.zeros(count, dtype=torch.int32, device=d)
trc, _ = timed(lambda: dev.compress_blocks_dev(ctx, src, off, ln, 4096, comp, coff, clen, prefix=t_dic, warm=dl.WARM_JENKINS))
trd, _ = timed(lambda: dev.decompress_blocks_dev(ctx, comp, coff, clen, out, off, ln32, olen32, st, dictionary=t_dic))
assert torch.equal(out[:tot], src)
print("raw blocks device-resident: compress %.2f GB/s (%.2f M msgs/s), decompress %.2f GB/s (%.2f M msgs/s)"
      % (tot / trc / 1e9, count / trc / 1e6, tot / trd / 1e9, count / trd / 1e6), flush=True)

# crossover: the same 256 MiB as frames of one size, batch call against a loop of single-frame calls (host to host)
total = 256 << 20
mixed = corpus.log(5, total).tobytes()
print("crossover (log text, 256 MiB, default options = linked 4 MiB blocks, and independent 64 KiB blocks):", flush=True)
for indep, mbs in ((False, 4194304), (True, 65536)):
    for fs in (64 << 10, 256 << 10, 1 << 20, 4 << 20, 16 << 20, 64 << 20):
        parts = [mixed[i:i + fs] for i in range(0, total, fs)]
        tb, fr = timed(lambda: dl.compressBuffers(parts, None, mbs, indep, ctx=ctx), 2)
        ts, fr1 = timed(lambda: [dl.compressBuffer(p, None, mbs, indep, ctx=ctx) for p in parts], 2)
        assert fr == fr1
        tbd, _ = timed(lambda: dl.decompressBuffers(fr, ctx=ctx), 2)
        tsd, _ = timed(lambda: [dl.decompressBuffer(f, ctx=ctx) for f in fr], 2)
        print("  indep=%d frame %6d KiB x %5d: compress batch %.2f / single %.2f GB/s, decompress batch %.2f / single %.2f GB/s"
              % (indep, fs >> 10, len(parts), total / tb / 1e9, total / ts / 1e9, total / tbd / 1e9, total / tsd / 1e9), flush=True)
