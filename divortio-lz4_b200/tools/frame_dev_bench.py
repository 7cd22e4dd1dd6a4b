"""Single frames in device memory against the host single-frame calls.  For each shape it times
  compress_tensor / decompress_tensor (device-resident: CUDA tensor in, CUDA tensor out), and
  dlz4_frame_compress / dlz4_frame_decompress between page-locked host buffers (the PCIe path),
and checks that both give the same frame and the input back.  It also times, separately, the parts of the device calls that
are not compression or decoding: the device-to-device staging copy of a frame, and frame_info_dev (staging copy + header
copy + k_fd_parse's one-thread walk of the block table + one synchronisation), whose difference is the walk.
Shapes: 1 GiB MIXED in independent 64 KiB blocks, 256 MiB log text in the reference's default frame (linked 4 MiB blocks),
64 MiB log text in linked 64 KiB blocks.  Rates are GB/s of uncompressed bytes, best of `reps` runs; inputs are larger than L2.
The first line names the card, its power limit and SM clocks, read in the same run.
Usage: python divortio-lz4_b200/tools/frame_dev_bench.py [reps] [out.txt]   (default 5; the report also goes to out.txt)"""
import ctypes as C
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

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
out_path = sys.argv[2] if len(sys.argv) > 2 else None
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True)
say("card (name, power limit, SM clock, max SM clock): %s" % q.stdout.strip())
ctx = dl.default_context(0)
L = dl.api.lib()
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


SHAPES = [
    ("1 GiB MIXED, independent 64 KiB blocks", lambda: corpus.mixed(1, 1 << 30), dict(maxBlockSize=65536, blockIndependence=True)),
    ("256 MiB log, default frame (linked 4 MiB)", lambda: corpus.log(2, 256 << 20), dict()),
    ("64 MiB log, linked 64 KiB blocks", lambda: corpus.log(3, 64 << 20), dict(maxBlockSize=65536)),
]

say("%-44s %10s %10s %10s %10s %8s | %10s %10s %10s" % ("shape", "c dev", "c host", "d dev", "d host", "ratio", "stage",
                                                      "info_dev", "walk~"))
for name, make, kw in SHAPES:
    data = make()
    n = data.size
    h_in = pinned(n)
    h_in[:] = data
    t_in = torch.from_numpy(data).to(cuda)
    opts = dl.api.frame_opts(**kw)
    cap = dl.frame_bound(n)
    h_frame = pinned(cap)
    flen = C.c_uint64(0)

    def host_compress():
        ctx.check(L.dlz4_frame_compress(ctx.handle, h_in.ctypes.data, n, None, 0, C.byref(opts), h_frame.ctypes.data, cap, C.byref(flen)))
        return int(flen.value)

    t_ch, fl = best(host_compress)
    t_cd, f_dev = best(lambda: dev.compress_tensor(t_in, **kw))
    assert f_dev.numel() == fl and np.array_equal(f_dev.cpu().numpy(), h_frame[:fl]), name
    h_out = pinned(n)
    olen = C.c_uint64(0)

    def host_decompress():
        ctx.check(L.dlz4_frame_decompress(ctx.handle, h_frame.ctypes.data, fl, None, 0, 1, h_out.ctypes.data, n, C.byref(olen)))
        return int(olen.value)

    t_dh, ol = best(host_decompress)
    assert ol == n and np.array_equal(h_out, data), name
    t_dd, out = best(lambda: dev.decompress_tensor(f_dev))
    assert torch.equal(out, t_in), name
    del out
    t_stage, _ = best(lambda: f_dev.clone())
    t_info, info = best(lambda: dev.frame_info_dev(ctx, f_dev))
    gb = n / 1e9
    say("%-44s %10.1f %10.1f %10.1f %10.1f %8.3f | %8.3fms %8.3fms %8.3fms   (%d blocks)" % (
        name, gb / t_cd, gb / t_ch, gb / t_dd, gb / t_dh, n / fl, t_stage * 1e3, t_info * 1e3, (t_info - t_stage) * 1e3,
        info.nblocks))
    del t_in, f_dev
    torch.cuda.empty_cache()

say("c/d dev: compress_tensor / decompress_tensor, GB/s;  c/d host: dlz4_frame_compress / dlz4_frame_decompress between "
    "page-locked buffers, GB/s")
say("stage: device-to-device copy of the frame;  info_dev: frame_info_dev (stage + header + k_fd_parse walk + sync);  "
    "walk~: info_dev - stage")
if out_path:
    with open(out_path, "w") as fh:
        fh.write("\n".join(lines) + "\n")
