"""GPU parity, concatenated frames in device memory: dlz4_frames_compress_dev / dlz4_frames_info_dev / dlz4_frames_decompress_dev
and compress_tensor_frames / decompress_tensor_frames against the oracle, the single-frame calls and the host frame loop
(dlz4_frames_info / dlz4_frames_decompress), byte for byte and status for status, on both decode routes.  -m gpu."""
import ctypes as C

import numpy as np
import pytest

import oracle
import test_gpu_decode_differential as dd
import test_gpu_frame_batch as fb
import test_gpu_frame_dev as fd
from conftest import GOLDEN_OPTS, edge_corpora, golden_inputs

pytestmark = pytest.mark.gpu

B64 = 65536
M4 = 4194304
E_OUTPUT_TOO_SMALL, E_MALFORMED, E_BAD_MAGIC, E_CONTENT_CHECKSUM, E_INVALID_ARG, E_TOO_LARGE = 1, 2, 5, 7, 20, 21


@pytest.fixture(scope="module")
def dl():
    import divortio_lz4_b200 as m
    m.default_context()
    return m


@pytest.fixture(scope="module")
def ctxs(dl):
    """The decode routes: "default" (frames below 4 MiB of max_decoded in warp groups, larger ones alone); "large": every
    frame alone through frame_decode; "warp": every frame that fits in a warp group, with a 64 KiB group budget so a
    sequence takes several groups; "small" / "chain": every frame alone, with the single-frame decode knobs of
    test_gpu_frame_dev (jump decoder for every frame / never)."""
    return {"default": dl.default_context(),
            "large": fd._ctx(dl, DLZ4_FRAMES_WARP_MAX_KIB="0"),
            "warp": fd._ctx(dl, DLZ4_FRAMES_WARP_MAX_KIB=str(1 << 40), DLZ4_FRAMES_GROUP_KIB="64"),
            "small": fd._ctx(dl, DLZ4_FRAMES_WARP_MAX_KIB="0", DLZ4_SEG_MIN_KIB="16", DLZ4_JUMP_MIN_KIB="0"),
            "chain": fd._ctx(dl, DLZ4_FRAMES_WARP_MAX_KIB="0", DLZ4_JUMP_MIN_KIB=str(1 << 30))}


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream or 1)


# ================================================================================ 1. compress parity
def _compress_dev(dl, ctx, data, frame_bytes, dictionary, kw, bc, offset=0):
    import torch
    src = fd._gpu(data, offset)
    d = fd._gpu(dictionary, offset) if dictionary else None
    k = max(1, -(-len(data) // frame_bytes))
    cap = sum(dl.frame_bound(min(frame_bytes, len(data) - i * frame_bytes)) for i in range(k)) if data else dl.frame_bound(0)
    dst = torch.empty(cap + offset, dtype=torch.uint8, device="cuda")[offset:]
    off = (C.c_uint64 * (k + 1))()
    n, nf = C.c_uint64(0), C.c_uint32(0)
    st = dl.api.lib().dlz4_frames_compress_dev(ctx.handle, fd._ptr(src), len(data), frame_bytes, fd._ptr(d), len(dictionary or b""),
                                               C.byref(fd._opts(dl, kw, bc)), fd._ptr(dst), cap, off, C.byref(n), C.byref(nf), _stream())
    assert st == 0, st
    assert nf.value == k
    return dst[:n.value].cpu().numpy().tobytes(), list(off[:k + 1])


def _spans(data, frame_bytes):
    return [data[i:i + frame_bytes] for i in range(0, len(data), frame_bytes)] or [data[:0]]


def _check_compress(dl, ctx, data, frame_bytes, dictionary=None, bc=False, offset=0, **kw):
    from divortio_lz4_b200 import device
    kw = fd._kw(**kw)
    got, off = _compress_dev(dl, ctx, data, frame_bytes, dictionary, kw, bc, offset)
    want = [fb._oracle_frame(bytes(s), dictionary, kw, bc) for s in _spans(data, frame_bytes)]
    assert got == b"".join(want), (len(data), frame_bytes, kw, bc, offset)
    assert off == list(np.concatenate([[0], np.cumsum([len(w) for w in want])]))
    d = fd._gpu(dictionary) if dictionary else None
    single = []
    for s in _spans(data, frame_bytes):
        import torch
        dst = torch.empty(dl.frame_bound(len(s)), dtype=torch.uint8, device="cuda")
        single.append(dst[:device.frame_compress_dev(ctx, fd._gpu(s), dst, fd._opts(dl, kw, bc), d)].cpu().numpy().tobytes())
    assert got == b"".join(single)
    return got


@pytest.mark.parametrize("opts", sorted(GOLDEN_OPTS))
@pytest.mark.parametrize("bc", [False, True])
def test_compress_parity_edge_golden_and_corpus_inputs(dl, opts, bc):
    from divortio_lz4_b200 import corpus
    ctx = dl.default_context()
    kw = fb._kw(GOLDEN_OPTS[opts])
    big = corpus.mixed(71, (5 << 20) // 2 + 17).tobytes()
    for data in list(edge_corpora().values()) + list(golden_inputs().values()) + [b"", big]:
        for frame_bytes in (1 << 20, 100003):                     # (100003: no multiple of any block size)
            _check_compress(dl, ctx, data, frame_bytes, None, bc, **kw)
    # frame_bytes >= src_len: compress_tensor's frame
    from divortio_lz4_b200 import device
    got, off = _compress_dev(dl, ctx, big, len(big), None, kw, bc)
    assert got == device.compress_tensor(fd._gpu(big), None, blockChecksum=bc, **kw).cpu().numpy().tobytes()
    assert off == [0, len(got)]
    assert _compress_dev(dl, ctx, b"", 7, None, kw, bc)[0] == fb._oracle_frame(b"", None, kw, bc)


def test_compress_parity_with_dictionaries(dl):
    from divortio_lz4_b200 import corpus
    ctx = dl.default_context()
    msgs = corpus.jsonmsgs(4, 0, 100).tobytes()[:300000]
    for dic in (corpus.json_dictionary(44).tobytes(), corpus.jsonmsgs(45, 0, 40).tobytes()[:100000], b"tiny"):
        for indep in (False, True):
            for mbs in (B64, M4):
                _check_compress(dl, ctx, msgs, 100003, dic, False, maxBlockSize=mbs, blockIndependence=indep, contentChecksum=True)


def test_compress_arguments(dl):
    import torch
    from divortio_lz4_b200 import device
    ctx = dl.default_context()
    L = dl.api.lib()
    src = fd._gpu(b"x" * 1000)
    dst = torch.empty(4096, dtype=torch.uint8, device="cuda")
    n, k = C.c_uint64(0), C.c_uint32(0)
    o = dl.api.frame_opts()

    def call(frame_bytes, cap):
        return L.dlz4_frames_compress_dev(ctx.handle, src.data_ptr(), 1000, frame_bytes, None, 0, C.byref(o), dst.data_ptr(), cap,
                                          None, C.byref(n), C.byref(k), _stream())
    assert call(0, 4096) == E_INVALID_ARG
    assert call(0x7FFF0000, 4096) == E_TOO_LARGE
    need = 2 * dl.frame_bound(500)
    assert call(500, need - 1) == E_OUTPUT_TOO_SMALL
    assert call(500, need) == 0 and k.value == 2
    with pytest.raises(ValueError):
        device.compress_tensor_frames(torch.zeros(8, dtype=torch.uint8))
    with pytest.raises(ValueError):
        device.decompress_tensor_frames(torch.zeros(8, dtype=torch.uint8))
    with pytest.raises(ValueError):
        device.compress_tensor_frames(torch.zeros(8, 8, dtype=torch.uint8, device="cuda").t())


# ================================================================================ 2. full size
def test_four_and_a_half_gib(dl):
    import torch
    from divortio_lz4_b200 import corpus, device, sharded
    ctx = dl.default_context()
    n = (9 << 30) // 2
    data = corpus.mixed(72, n)
    t = torch.from_numpy(data).cuda()
    spans = sharded.frame_spans(n)
    assert len(spans) == 5
    # independent blocks with both checksums: what compress_sharded writes with one rank
    f = device.compress_tensor_frames(t, maxBlockSize=B64, blockIndependence=True, contentChecksum=True, blockChecksum=True)
    out = np.empty(sum(dl.frame_bound(hi - lo) for lo, hi in spans) + 4096, dtype=np.uint8)
    total = sharded.compress_sharded(data, out, B64, True, True, True, comm=sharded.LocalComm(), backend=sharded.GpuBackend(ctx))
    assert total == f.numel() and torch.equal(f, torch.from_numpy(out[:total]).cuda())
    del out
    back, frames = device.decompress_tensor_frames(f, verifyBlockChecksums=True)
    assert frames == 5 and torch.equal(back, t)
    del back
    # the host frame loop reads the same bytes
    host = f.cpu().numpy()
    dst = np.empty(n + 64, dtype=np.uint8)
    got, cnt = C.c_uint64(0), C.c_uint32(0)
    st = dl.api.lib().dlz4_frames_decompress(ctx.handle, host.ctypes.data, host.size, None, 0, 3, dst.ctypes.data, n, C.byref(got),
                                             C.byref(cnt))
    assert (st, got.value, cnt.value) == (0, n, 5) and np.array_equal(dst[:n], data)
    del host, dst, f
    # the default linked frame: per-span compress_tensor, the last span against the oracle
    g = device.compress_tensor_frames(t)
    parts = [device.compress_tensor(t[lo:hi]) for lo, hi in spans]
    assert torch.equal(g, torch.cat(parts))
    assert parts[-1].cpu().numpy().tobytes() == oracle.compress_buffer(data[spans[-1][0]:])
    del parts
    back, frames = device.decompress_tensor_frames(g)
    assert frames == 5 and torch.equal(back, t)


# ================================================================================ 3-5. decode parity, routes, info
def _skippable(nibble, payload):
    return (0x184D2A50 | nibble).to_bytes(4, "little") + len(payload).to_bytes(4, "little") + payload


def _host_frames(dl, ctx, data, dictionary, flags, cap):
    out = np.zeros(max(cap, 1) + 64, dtype=np.uint8)
    a = np.frombuffer(data, dtype=np.uint8) if data else np.zeros(1, dtype=np.uint8)
    d = np.frombuffer(dictionary, dtype=np.uint8) if dictionary else None
    n, k = C.c_uint64(0), C.c_uint32(0)
    st = dl.api.lib().dlz4_frames_decompress(ctx.handle, a.ctypes.data, len(data), d.ctypes.data if d is not None else None,
                                             len(dictionary or b""), flags, out.ctypes.data, cap, C.byref(n), C.byref(k))
    return st, n.value, k.value, out[:n.value].tobytes()


def _dev_frames(dl, ctx, data, dictionary, flags, cap, offset=0):
    import torch
    src = fd._gpu(data if data else b"\0", offset)
    d = fd._gpu(dictionary, offset) if dictionary else None
    dst = torch.empty(cap + offset, dtype=torch.uint8, device="cuda")[offset:]
    n, k = C.c_uint64(0), C.c_uint32(0)
    st = dl.api.lib().dlz4_frames_decompress_dev(ctx.handle, src.data_ptr(), len(data), fd._ptr(d), len(dictionary or b""), flags,
                                                 fd._ptr(dst), cap, C.byref(n), C.byref(k), _stream())
    assert st < 20, st
    return st, n.value, k.value, dst[:n.value].cpu().numpy().tobytes()


def _info_pair(dl, ctx, data):
    a = np.frombuffer(data, dtype=np.uint8) if data else np.zeros(1, dtype=np.uint8)
    hm, hk, dm, dk = C.c_uint64(0), C.c_uint32(0), C.c_uint64(0), C.c_uint32(0)
    hs = dl.api.lib().dlz4_frames_info(a.ctypes.data, len(data), C.byref(hm), C.byref(hk))
    t = fd._gpu(data if data else b"\0", 5)
    ds = dl.api.lib().dlz4_frames_info_dev(ctx.handle, t.data_ptr(), len(data), C.byref(dm), C.byref(dk), _stream())
    return (hs, hm.value, hk.value), (ds, dm.value, dk.value)


def _sequences(dl, kats):
    """(tag, [pieces], dictionary): concatenations of frames of every writer with skippable frames, and error cases."""
    rng = np.random.RandomState(140)
    valid = fd._valid_frames(dl, kats)[::3]
    skips = [_skippable(i, bytes(rng.randint(0, 256, i * 3, dtype=np.uint8))) for i in range(16)]
    mixed = [skips[0]]
    for i, f in enumerate(valid):
        mixed.append(f)
        if i % 4 == 0:
            mixed.append(skips[(i // 4) % 16])
    mixed += skips[1:] + [_skippable(15, b"")]
    yield "writers_and_skippable", mixed, None
    routes = [fr for _, fr in fd._route_frames() if not fr.dictionary]
    yield "routes", [f.bytes() for f in routes] + [_skippable(3, b"xyz")] + [f.bytes() for f in routes[::-1]], None
    dic_frames = [fr for _, fr in fd._route_frames() if fr.dictionary]
    for fr in dic_frames:
        yield "dict", [fr.bytes(), _skippable(7, b""), fr.bytes()], fr.dictionary
    good = [oracle.compress_buffer(corpus_bytes(i), None, B64, i % 2 == 1, True) for i in range(5)]
    frames, _ = fb._error_frames(dl, rng)
    bad = [f for f in frames if f not in good][::4]
    for k, b in enumerate(bad):
        yield "bad%d_first" % k, [b] + good, None
        yield "bad%d_middle" % k, good[:2] + [b] + good[2:], None
        yield "bad%d_last" % k, good + [b], None
    for t in (1, 2, 3):
        yield "trailing%d" % t, good + [b"\x04\x22\x4d"[:t]], None
    sk = _skippable(9, b"payload!")
    yield "truncated_skippable_header", good + [sk[:6]], None
    yield "truncated_skippable_payload", good + [sk[:-2]], None
    cc_bad = bytearray(good[1])
    cc_bad[-1] ^= 0x5A                                                # content checksum error in frame 1 ...
    yield "checksum_then_malformed", [good[0], bytes(cc_bad), good[2][:len(good[2]) // 2]], None   # ... then a malformed frame 2


def corpus_bytes(i):
    from divortio_lz4_b200 import corpus
    return corpus.log(150 + i, 20000 + 7919 * i).tobytes()


def _caps(dl, ctx, data, pieces):
    a = np.frombuffer(data, dtype=np.uint8)
    total, k = C.c_uint64(0), C.c_uint32(0)
    dl.api.lib().dlz4_frames_info(a.ctypes.data, len(data), C.byref(total), C.byref(k))
    caps = {int(total.value), max(int(total.value) - 1, 0)}
    mds = []
    for p in pieces:
        try:
            mds.append(int(dl.frame_info(p).max_decoded))
        except dl.LZ4Error:
            pass
    if len(mds) >= 3:
        h = len(mds) // 2
        caps.add(sum(mds[:h]) + mds[h] // 2)                      # binds in the middle frame
    return sorted(caps)


@pytest.mark.parametrize("flags", list(range(8)))
def test_decode_parity_with_the_host_frame_loop(dl, ctxs, kats, flags):
    for tag, pieces, dic in _sequences(dl, kats):
        data = b"".join(pieces)
        for cap in _caps(dl, ctxs["default"], data, pieces):
            want = _host_frames(dl, ctxs["default"], data, dic, flags, cap)
            for name, ctx in ctxs.items():
                got = _dev_frames(dl, ctx, data, dic, flags, cap)
                assert got[:3] == want[:3] and got[3] == want[3], (tag, name, flags, cap, got[:3], want[:3])


def test_error_sequences_report_the_first_failing_frame(dl, kats):
    seqs = {tag: (pieces, dic) for tag, pieces, dic in _sequences(dl, kats)}
    ctx = dl.default_context()
    pieces, _ = seqs["checksum_then_malformed"]
    st, n, k, _ = _dev_frames(dl, ctx, b"".join(pieces), None, 1, 1 << 20)
    assert (st, k) == (E_CONTENT_CHECKSUM, 1) and n == 20000
    st, n, k, _ = _dev_frames(dl, ctx, b"".join(pieces), None, 0, 1 << 20)
    assert (st, k) == (E_MALFORMED, 2)
    for t in (1, 2, 3):
        assert _dev_frames(dl, ctx, b"".join(seqs["trailing%d" % t][0]), None, 1, 1 << 20)[:3:2] == (E_BAD_MAGIC, 5)


def test_info_equals_the_host_call(dl, ctxs, kats):
    ctx = ctxs["default"]
    for tag, pieces, _ in _sequences(dl, kats):
        want, got = _info_pair(dl, ctx, b"".join(pieces))
        assert got == want, tag
    three = oracle.compress_buffer(b"abc" * 50) + _skippable(2, b"skip") + oracle.compress_buffer(b"defg" * 40, None, B64, True, True)
    for k in range(len(three) + 1):
        want, got = _info_pair(dl, ctx, three[:k])
        assert got == want, k
    assert _info_pair(dl, ctx, three)[1] == (0, 310, 2)


# ================================================================================ 6. many small frames
def test_one_hundred_thousand_json_frames(dl):
    import torch
    from divortio_lz4_b200 import corpus, device
    blob = corpus.jsonmsgs(160, 0, 100000)
    msgs = [blob[i * 4096:(i + 1) * 4096].tobytes() for i in range(100000)]
    for cc in (False, True):
        frames = dl.compressBuffers(msgs, contentChecksum=cc)
        data = torch.frombuffer(bytearray(b"".join(frames)), dtype=torch.uint8).cuda()
        out, n = device.decompress_tensor_frames(data)
        assert n == 100000
        assert out.cpu().numpy().tobytes() == b"".join(msgs)


# ================================================================================ 7. caller memory and streams
def test_unaligned_caller_memory(dl):
    from divortio_lz4_b200 import corpus
    ctx = dl.default_context()
    data = corpus.log(161, 700001).tobytes()
    dic = corpus.json_dictionary(162).tobytes()
    for offset in (1, 3, 7):
        for kw in (dict(), dict(maxBlockSize=B64, blockIndependence=True, contentChecksum=True),
                   dict(maxBlockSize=B64, contentChecksum=True)):
            for frame_bytes in (200000, 200003):                      # checksum chains on aligned and unaligned spans
                f = _check_compress(dl, ctx, data, frame_bytes, dic, True, offset, **kw)
                assert _dev_frames(dl, ctx, f, dic, 3, len(data), offset) == (0, len(data), -(-len(data) // frame_bytes), data)


def test_tensors_that_end_flush_with_their_allocation(dl):
    import torch
    from divortio_lz4_b200 import corpus, device
    for n, kw in (((1 << 20) + 512, dict(contentChecksum=True)), (300 * 1024, dict(maxBlockSize=B64, blockIndependence=True,
                                                                                  contentChecksum=True))):
        data = corpus.mixed(163, n).tobytes()
        assert n % 512 == 0
        src = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        f = device.compress_tensor_frames(src, frame_max=n // 3 + 1, **kw)
        want = b"".join(fb._oracle_frame(s, None, fd._kw(**kw), False) for s in _spans(data, n // 3 + 1))
        assert f.cpu().numpy().tobytes() == want
        pad = (-len(want)) % 512
        buf = torch.zeros(len(want) + pad, dtype=torch.uint8, device="cuda")
        buf[pad:] = f
        frame = buf[pad:]
        assert frame.data_ptr() + frame.numel() == buf.data_ptr() + buf.numel()
        out, k = device.decompress_tensor_frames(frame)
        assert k == 3 and out.cpu().numpy().tobytes() == data


def test_non_default_stream(dl):
    import torch
    from divortio_lz4_b200 import corpus, device
    data = corpus.log(164, (24 << 20) + 11).tobytes()
    plain = (np.frombuffer(data, dtype=np.uint8) ^ 0x5A).tobytes()
    want = b"".join(oracle.compress_buffer(s, None, B64, False, True) for s in _spans(plain, 5 << 20))
    base = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        x = torch.bitwise_xor(base, 0x5A)                           # queued on s, not finished when the call starts
        f = device.compress_tensor_frames(x, None, B64, False, True, frame_max=5 << 20)
        g = f.clone()
        out, k = device.decompress_tensor_frames(g)
        got_f, got = f.cpu().numpy().tobytes(), out.cpu().numpy().tobytes()
    s.synchronize()
    assert got_f == want and k == 5
    assert got == plain
