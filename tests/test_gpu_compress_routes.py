"""GPU parity, compression routes: launch_compress (csrc/api_launch.inc) picks a kernel from the batch's largest block, its
prefix and table, its block count and whether its blocks tile one range uniformly.  Every case here drives one route through
the public calls, checks under torch.profiler which kernels ran, and compares every block with the oracle:

  k_parse_pw + k_encode_blocks   fresh blocks <= 64 KiB, at most 2^20 of them; sliced when the match records of one launch would
                                 pass kRecLaunchBytes (one 64 KiB block among 300 000 small ones, 16 GiB of 64 KiB blocks)
  k_compress_fresh16h            the same blocks, more than 2^20 of them (also a dense chunk of the packed pipeline)
  k_compress_overlay             blocks <= 4096 bytes behind a prefix and table (several chunks of the packed pipeline)
  k_compress_generic32           "unknown" largest block (0xFFFFFFFF), ragged or non-power-of-two blocks > 64 KiB, uniform blocks
                                 ending past 2 GiB of the base, blocks > 4096 bytes behind a prefix

Batches too large to hold twice on the host are compared by comp_len and per-block xxh32; the rest byte for byte.  -m gpu."""
import contextlib
import os

import numpy as np
import pytest

import oracle
from conftest import edge_corpora
from test_gpu_blocks import _fuzz_block, _pack

pytestmark = pytest.mark.gpu

SPLIT = 1 << 20                      # kMaxSplitBlocks: the split path's block limit per launch
GIB = 1 << 30
FINDER = ("k_parse_pw", "k_encode_blocks")
OTHERS = ("k_compress_fresh16h", "k_compress_overlay", "k_compress_segments", "k_compress_generic32")


@pytest.fixture(scope="module")
def dl():
    import torch
    import divortio_lz4_b200 as m
    m.default_context()
    torch.zeros(1, device="cuda")    # torch's CUDA state exists before the first profiler session
    return m


class env_ctx:
    """Knobs such as DLZ4_CHUNK_MIB are read once, by dlz4_init: the default context is replaced by one created under the
    wanted environment and dropped again on exit."""

    def __init__(self, **knobs):
        self.new = {k: (None if v is None else str(v)) for k, v in knobs.items()}

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.new}
        self._set(self.new)

    def __exit__(self, *a):
        self._set(self.old)

    @staticmethod
    def _set(values):
        for k, v in values.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        from divortio_lz4_b200 import api
        api._default.clear()                                    # (contexts other modules still hold stay alive)


def _kernel_names(prof):
    names = [e.name for e in prof.events()]
    try:
        names += [e.name() for e in prof.profiler.kineto_results.events()]
    except AttributeError:
        pass
    return names


@contextlib.contextmanager
def route(expect, absent=()):
    """Asserts that every kernel named in `expect` ran inside the block and none named in `absent` did."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        yield
        torch.cuda.synchronize()
    names = _kernel_names(prof)
    ran = sorted({n for n in names if n.startswith(("k_", "void k_", "_Z"))})
    for k in expect:
        assert any(k in n for n in names), ("expected kernel did not run", k, ran)
    for k in absent:
        assert not any(k in n for n in names), ("unexpected kernel ran", k, ran)


def _assert_same_blocks(got, want, what):
    """Per-block equality of two (dst, dst_off, comp_len) results: lengths, then the xxh32 of every block's bytes."""
    dst, doff, clen = got
    odst, odoff, oclen = want
    assert np.array_equal(clen, oclen), (what, np.nonzero(clen != oclen)[0][:10])
    bad = np.nonzero(oracle.xxh32_batch(dst, doff, clen) != oracle.xxh32_batch(odst, odoff, oclen))[0]
    assert not bad.size, (what, "blocks differ from the oracle", bad[:10])


def _assert_same_bytes(got, want, what):
    dst, doff, clen = got
    odst, odoff, oclen = want
    assert np.array_equal(clen, oclen), (what, np.nonzero(clen != oclen)[0][:10])
    bad = [i for i in range(len(clen)) if not np.array_equal(dst[int(doff[i]):int(doff[i]) + int(clen[i])],
                                                             odst[int(odoff[i]):int(odoff[i]) + int(oclen[i])])]
    assert not bad, (what, "blocks differ from the oracle", bad[:10])


def _strided_layout(ln):
    bound = (ln.astype(np.uint64) + ln.astype(np.uint64) // 255 + 16 + 15) & ~np.uint64(15)
    doff = np.zeros(len(ln), dtype=np.uint64)
    doff[1:] = np.cumsum(bound)[:-1]
    return doff, int(bound.sum())


def _device_compress(dl, src, off, ln, max_len, **kw):
    """compress_blocks_dev on host arrays (uploaded), strided output; returns host (dst, dst_off, comp_len)."""
    import torch
    from divortio_lz4_b200 import device as dev
    ctx = dl.default_context()
    t = lambda a: torch.from_numpy(np.require(a, requirements=["C", "W"])).cuda()
    doff, total = _strided_layout(ln)
    dst = torch.zeros(total + 16, dtype=torch.uint8, device="cuda")
    clen = torch.zeros(len(ln), dtype=torch.int32, device="cuda")
    dev.compress_blocks_dev(ctx, t(src), t(off.view(np.int64)), t(ln.view(np.int32)), max_len, dst, t(doff.view(np.int64)), clen, **kw)
    torch.cuda.synchronize()
    return dst.cpu().numpy(), doff, clen.cpu().numpy().view(np.uint32)


def _packed_as_strided(pdst, pclen):
    doff = np.zeros(len(pclen), dtype=np.uint64)
    doff[1:] = np.cumsum(pclen.astype(np.uint64))[:-1]
    return pdst, doff, pclen


@pytest.fixture(scope="module")
def base():
    """~24 MiB of structured data: fuzz blocks (copies at every distance, runs, periods, noise, words) back to back.  Blocks
    of the batches below are slices of it, tiled as far as a batch needs."""
    rng = np.random.RandomState(2026)
    return np.frombuffer(b"".join(_fuzz_block(rng, int(n)) for n in rng.randint(1, 65537, size=720)), dtype=np.uint8)


def _slices(base, ln, rng, max_gap=8):
    """Ascending, disjoint blocks of the given lengths at odd gaps in a tiling of `base`: (src, off)."""
    gap = rng.randint(0, max_gap, size=len(ln)).astype(np.uint64)
    step = ln.astype(np.uint64) + gap
    off = np.cumsum(step) - ln.astype(np.uint64)
    total = int(off[-1]) + int(ln[-1]) + 16
    return np.resize(base, total), off


FUZZ_CLASSES = [0, 1, 4, 5, 11, 12, 13, 14, 31, 32, 33, 63, 64, 65, 95, 96, 97, 111, 112, 113, 127, 128, 129, 143, 144, 145,
                4095, 4096, 4097]


@pytest.fixture(scope="module")
def boundary_batch(dl, base):
    """2^20 + 2^18 blocks of 0..2000 bytes (most below 300), every length class of the fuzz test 40 times, and 400 blocks of
    8..60 KiB: the 16-bit-position blocks (Tab16 / TabG16) that force the next small block of a warp to clear its table.  The
    longest block stays below 64 KiB."""
    rng = np.random.RandomState(20)
    n = SPLIT + SPLIT // 4
    ln = np.where(rng.rand(n) < 0.7, rng.randint(0, 301, size=n), rng.randint(0, 2001, size=n)).astype(np.uint32)
    pos = rng.choice(n, size=len(FUZZ_CLASSES) * 40 + 400, replace=False)
    ln[pos[:len(FUZZ_CLASSES) * 40]] = np.tile(FUZZ_CLASSES, 40)
    ln[pos[len(FUZZ_CLASSES) * 40:]] = rng.randint(8192, 61441, size=400)
    src, off = _slices(base, ln, rng)
    return src, off, ln, oracle.compress_blocks(src, off, ln)


def _head(res, k):
    dst, doff, clen = res
    return dst, doff[:k], clen[:k]


@pytest.mark.parametrize("n", [SPLIT, SPLIT + 1])
def test_split_limit_strided_and_device_calls(dl, boundary_batch, n):
    """Exactly 2^20 blocks run the match finder; one more runs k_compress_fresh16h (every warp wraps its 4-bit small-block epoch
    many times, shared-memory and L2-table warps alike).  Both give the oracle's bytes."""
    src, off, ln, want = boundary_batch
    off, ln = off[:n], ln[:n]
    expect, absent = (FINDER, ("k_compress_fresh16h",)) if n <= SPLIT else (("k_compress_fresh16h",), FINDER)
    with route(expect, absent):
        got = dl.compress_blocks(src, off, ln)
    _assert_same_blocks(got, _head(want, n), ("strided", n))
    with route(expect, absent):
        got = _device_compress(dl, src, off, ln, int(ln.max()))
    _assert_same_blocks(got, _head(want, n), ("device", n))


def test_packed_pipeline_dense_chunk_over_split_limit(dl, boundary_batch):
    """The packed call with a chunk size that puts 2^20 + 1 blocks or more into the first of two chunks: that chunk runs
    k_compress_fresh16h with dense CTAs (7 chains each), the second the match finder."""
    src, off, ln, want = boundary_batch
    cum = np.cumsum(ln.astype(np.uint64))
    chunk_mib = -(-int(cum[SPLIT]) // (1 << 20))
    assert int(cum[-1]) > chunk_mib << 20                  # a second chunk exists
    with env_ctx(DLZ4_CHUNK_MIB=chunk_mib):
        with route(("k_compress_fresh16h",) + FINDER):
            pdst, _, pclen = dl.compress_blocks(src, off, ln, packed=True)
    _assert_same_blocks(_packed_as_strided(pdst, pclen), want, "packed")


@pytest.fixture(scope="module")
def ragged_batch(dl, base):
    """About 300 000 blocks of 0..400 bytes and one of 65 536 (which sets the match-record stride of the whole batch)."""
    rng = np.random.RandomState(21)
    n = 300001
    ln = rng.randint(0, 401, size=n).astype(np.uint32)
    ln[:len(FUZZ_CLASSES) - 3] = FUZZ_CLASSES[:-3]
    ln[n // 2] = 65536
    src, off = _slices(base, ln, rng)
    return src, off, ln, oracle.compress_blocks(src, off, ln)


def test_ragged_batch_with_one_64k_block_block_calls(dl, ragged_batch):
    src, off, ln, want = ragged_batch
    absent = ("k_compress_fresh16h", "k_compress_generic32")
    with route(FINDER, absent):
        got = dl.compress_blocks(src, off, ln)
    _assert_same_bytes(got, want, "strided")
    with route(FINDER, absent):
        got = _device_compress(dl, src, off, ln, 65536)
    _assert_same_bytes(got, want, "device")
    with route(FINDER, absent):
        pdst, _, pclen = dl.compress_blocks(src, off, ln, packed=True)
    _assert_same_bytes(_packed_as_strided(pdst, pclen), want, "packed")


def test_ragged_batch_with_one_64k_block_frame_batch(dl, ragged_batch):
    """compressBuffers on the same messages: one frame each, every frame equal to the oracle's compressBuffer."""
    src, off, ln, _ = ragged_batch
    msgs = [src[int(o):int(o) + int(k)] for o, k in zip(off, ln)]
    with route(FINDER, ("k_compress_fresh16h",)):
        frames = dl.compressBuffers(msgs)
    bad = [i for i, m in enumerate(msgs) if frames[i] != oracle.compress_buffer(m)]
    assert not bad, ("frames differ from the oracle", bad[:10])


@pytest.fixture(scope="module")
def mixed_1g():
    from divortio_lz4_b200 import corpus
    return corpus.mixed(2, GIB)


def _tiled_reference(data, block, reps):
    """The oracle's comp_len and per-block xxh32 of `data` in blocks of `block` bytes, tiled `reps` times (blocks are
    independent, so a tensor of `reps` copies of `data` compresses to `reps` copies of them)."""
    off = np.arange(0, data.size, block, dtype=np.uint64)
    ln = np.full(len(off), block, dtype=np.uint32)
    odst, odoff, oclen = oracle.compress_blocks(data, off, ln)
    return np.tile(oclen, reps), np.tile(oracle.xxh32_batch(odst, odoff, oclen), reps)


def _device_tiled_compress(dl, mixed_1g, reps, block):
    """compress_blocks_dev over `reps` device copies of the 1 GiB buffer in blocks of `block` bytes, strided output.
    Returns (src, dst, dst_off, comp_len, off, len) as CUDA tensors."""
    import torch
    from divortio_lz4_b200 import device as dev
    ctx = dl.default_context()
    src = torch.from_numpy(mixed_1g).cuda().repeat(reps)
    nb = reps * GIB // block
    stride = (block + block // 255 + 16 + 15) & ~15
    idx = torch.arange(nb, dtype=torch.int64, device="cuda")
    off, ln = idx * block, torch.full((nb,), block, dtype=torch.int32, device="cuda")
    dst = torch.empty(nb * stride, dtype=torch.uint8, device="cuda")
    doff, clen = idx * stride, torch.zeros(nb, dtype=torch.int32, device="cuda")
    dev.compress_blocks_dev(ctx, src, off, ln, block, dst, doff, clen)
    torch.cuda.synchronize()
    return src, dst, doff, clen, off, ln


def _device_hashes(dl, dst, doff, clen):
    import torch
    from divortio_lz4_b200 import device as dev
    h = torch.zeros(clen.numel(), dtype=torch.int32, device="cuda")
    dev.xxh32_batch_dev(dl.default_context(), dst, doff, clen, h)
    return h.cpu().numpy().view(np.uint32)


def test_device_batch_16gib_of_64k_blocks(dl, mixed_1g):
    """262 144 blocks of 64 KiB (16 GiB) through compress_blocks_dev: the match finder in slices, each block equal to the
    oracle's; then decoded back on the device."""
    import torch
    from divortio_lz4_b200 import device as dev
    reps = 16
    with route(FINDER, ("k_compress_fresh16h", "k_compress_generic32")):
        src, dst, doff, clen, off, ln = _device_tiled_compress(dl, mixed_1g, reps, 65536)
    want_len, want_hash = _tiled_reference(mixed_1g, 65536, reps)
    assert np.array_equal(clen.cpu().numpy().view(np.uint32), want_len)
    assert np.array_equal(_device_hashes(dl, dst, doff, clen), want_hash)
    out = torch.empty_like(src)
    olen = torch.zeros_like(clen)
    status = torch.zeros(clen.numel(), dtype=torch.uint8, device="cuda")
    dev.decompress_blocks_dev(dl.default_context(), dst, doff, clen, out, off, ln, olen, status)
    torch.cuda.synchronize()
    assert int(status.max()) == 0 and torch.equal(olen, ln) and torch.equal(out, src)


def test_uniform_4m_blocks_ending_past_2gib(dl, mixed_1g):
    """768 uniform 4 MiB blocks of a 3 GiB tensor end past 0x7FFFFFF0 of the base: not the segment engine, one warp per block
    (k_compress_generic32), the oracle's bytes all the same."""
    with route(("k_compress_generic32",), ("k_compress_segments",) + FINDER):
        src, dst, doff, clen, off, ln = _device_tiled_compress(dl, mixed_1g, 3, 4 << 20)
    want_len, want_hash = _tiled_reference(mixed_1g, 4 << 20, 3)
    assert np.array_equal(clen.cpu().numpy().view(np.uint32), want_len)
    assert np.array_equal(_device_hashes(dl, dst, doff, clen), want_hash)


def test_unknown_max_block_len_on_small_blocks(dl):
    """max_block_len = 0xFFFFFFFF ("unknown", as the header allows) on blocks <= 64 KiB: k_compress_generic32, the oracle's
    bytes, on the edge corpora and a fuzz batch of every length class."""
    rng = np.random.RandomState(33)
    corp = edge_corpora()
    lens = FUZZ_CLASSES + [65535, 65536] + [int(x) for x in rng.randint(0, 2000, size=300)] + \
        [int(x) for x in rng.randint(2000, 65537, size=300)]
    items = list(corp.values()) + [_fuzz_block(rng, n) for n in lens]
    buf, off, ln = _pack(items)
    with route(("k_compress_generic32",), FINDER + ("k_compress_fresh16h",)):
        got = _device_compress(dl, buf, off, ln, 0xFFFFFFFF)
    _assert_same_bytes(got, oracle.compress_blocks(buf, off, ln), "unknown max_block_len")


def test_ragged_and_non_power_of_two_large_blocks(dl, base):
    """Blocks > 64 KiB that do not tile one range with one power-of-two size: ragged (65 537, 100 000, 262 143, 1 048 577 and
    random sizes, some small ones among them) at scattered, overlapping offsets, and uniform 100 000-byte blocks."""
    rng = np.random.RandomState(34)
    src = np.resize(base, 8 << 20)
    ln = np.array([65537, 100000, 262143, 1048577, 65537, 3, 4096, 65536] + [int(x) for x in rng.randint(65537, 2 << 20, size=24)],
                  dtype=np.uint32)
    off = np.array([rng.randint(0, src.size - int(k) + 1) for k in ln], dtype=np.uint64)
    with route(("k_compress_generic32",), ("k_compress_segments",) + FINDER):
        got = dl.compress_blocks(src, off, ln)
    _assert_same_bytes(got, oracle.compress_blocks(src, off, ln), "ragged")
    n = 80
    off = np.arange(n, dtype=np.uint64) * 100000 + 5
    ln = np.full(n, 100000, dtype=np.uint32)
    ln[-1] = 77777
    with route(("k_compress_generic32",), ("k_compress_segments",) + FINDER):
        got = dl.compress_blocks(src, off, ln)
    _assert_same_bytes(got, oracle.compress_blocks(src, off, ln), "uniform 100000")


@pytest.mark.parametrize("plen", [37, 4097, 65535, 65536])
def test_blocks_over_4k_behind_a_prefix(dl, base, plen):
    """Messages of 4097, 8192, 65 535 and 65 536 bytes behind a prefix, from the Jenkins-warmed or a primed table: too long for
    the overlay kernel, so k_compress_generic32 runs compress_block_warp over the split source (prefix, then message)."""
    rng = np.random.RandomState(plen)
    dic = np.ascontiguousarray(base[1000:1000 + plen])
    ln = np.array([4097, 8192, 65535, 65536] * 24, dtype=np.uint32)
    rng.shuffle(ln)
    src, off = _slices(base[200000:], ln, rng, max_gap=40)
    work = np.concatenate([dic, np.zeros(8, dtype=np.uint8)])
    primed = oracle.new_table()
    oracle.compress_block(dic, 0, dic.size, primed)
    for mode, (warm, init, otab) in {"jenkins": (dl.WARM_JENKINS, None, oracle.warm_table_jenkins(work, dic.size)),
                                     "primed": (dl.WARM_TABLE, primed, primed)}.items():
        with route(("k_compress_generic32",), ("k_compress_overlay",) + FINDER):
            got = dl.compress_blocks(src, off, ln, prefix=dic, warm=warm, init_table=init)
        _assert_same_bytes(got, oracle.compress_blocks_prefix(dic, otab, src, off, ln), (plen, mode))


def test_packed_pipeline_prefix_several_chunks(dl):
    """40 000 JSON messages of 4 KiB behind the 64 KiB dictionary, 16 MiB chunks: k_compress_overlay with dense CTAs on three
    lanes, each with its own table region; the packed stream equals the oracle's blocks back to back."""
    from divortio_lz4_b200 import corpus
    nmsg = 40000
    msgs = corpus.jsonmsgs(4, 100, nmsg)
    dic = corpus.json_dictionary(44)
    off = np.arange(nmsg, dtype=np.uint64) * 4096
    ln = np.full(nmsg, 4096, dtype=np.uint32)
    primed = oracle.new_table()
    oracle.compress_block(dic, 0, dic.size, primed)
    want = oracle.compress_blocks_prefix(dic, primed, msgs, off, ln)
    with env_ctx(DLZ4_CHUNK_MIB=16):
        with route(("k_compress_overlay",), ("k_compress_generic32",)):
            pdst, _, pclen = dl.compress_blocks(msgs, off, ln, prefix=dic, warm=dl.WARM_TABLE, init_table=primed, packed=True)
    _assert_same_bytes(_packed_as_strided(pdst, pclen), want, "packed prefix")


def test_refused_scratch_allocation_leaves_no_error_behind(dl):
    """A call whose scratch cannot be allocated fails with DLZ4_E_CUDA; the next call on the same context succeeds."""
    from divortio_lz4_b200 import api
    ctx = dl.default_context()
    src = np.frombuffer(b"refused allocation " * 40, dtype=np.uint8)
    off, ln = np.zeros(1, dtype=np.uint64), np.array([src.size], dtype=np.uint32)
    dst, doff, comp = np.zeros(2048, dtype=np.uint8), np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint32)
    # dst_bytes sizes the device scratch of the output: 1 PiB cannot be had
    st = api.lib().dlz4_compress_blocks(ctx.handle, src.ctypes.data, src.size, off.ctypes.data, ln.ctypes.data, 1, None, 0, 0, None,
                                        dst.ctypes.data, 1 << 50, doff.ctypes.data, comp.ctypes.data)
    assert st == api.E_CUDA
    got = dl.compress_blocks(src, off, ln)
    _assert_same_bytes(got, oracle.compress_blocks(src, off, ln), "after a refused allocation")
