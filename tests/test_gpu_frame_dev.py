"""GPU parity, single frames in device memory: dlz4_frame_compress_dev / dlz4_frame_info_dev / dlz4_frame_decompress_dev and
compress_tensor / decompress_tensor against the oracle and against the host-pointer calls, byte for byte and status for
status, on every compress and decode route.  -m gpu."""
import ctypes as C
import os
import types

import numpy as np
import pytest

import oracle
import test_gpu_decode_differential as dd
import test_gpu_frame_batch as fb
from conftest import GOLDEN_OPTS, edge_corpora, golden_inputs

pytestmark = pytest.mark.gpu

B64 = 65536
M4 = 4194304


@pytest.fixture(scope="module")
def dl():
    import divortio_lz4_b200 as m
    m.default_context()
    return m


def _ctx(dl, **env):
    """A context with some knobs set: they are read when the context is created."""
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


@pytest.fixture(scope="module")
def ctxs(dl):
    """default; "small": the segment engine from 16 KiB and the jump decoder for every frame; "chain": never the jump decoder
    (short linked frames go to k_decompress_chain, independent ones to the strided decode)."""
    return {"default": dl.default_context(),
            "small": _ctx(dl, DLZ4_SEG_MIN_KIB="16", DLZ4_JUMP_MIN_KIB="0"),
            "chain": _ctx(dl, DLZ4_JUMP_MIN_KIB=str(1 << 30))}


def _gpu(data, offset=0, slack=0):
    """bytes -> a uint8 CUDA tensor view at `offset` bytes into a larger tensor (slack bytes behind it)."""
    import torch
    buf = torch.full((offset + len(data) + slack,), 0xA5, dtype=torch.uint8, device="cuda")
    view = buf[offset:offset + len(data)]
    if len(data):
        view.copy_(torch.frombuffer(bytearray(data), dtype=torch.uint8))
    return view


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() else None


def _opts(dl, kw, bc):
    return dl.api.frame_opts(kw["maxBlockSize"], kw["blockIndependence"], kw["contentChecksum"], kw["addContentSize"], bc)


def _compress_dev(dl, ctx, data, dictionary, kw, bc, offset=0):
    from divortio_lz4_b200 import device
    src = _gpu(data, offset)
    d = _gpu(dictionary, offset) if dictionary else None
    import torch
    dst = torch.empty(dl.frame_bound(len(data)) + offset, dtype=torch.uint8, device="cuda")[offset:]
    n = device.frame_compress_dev(ctx, src, dst, _opts(dl, kw, bc), d)
    return dst[:n].cpu().numpy().tobytes()


def _kw(maxBlockSize=M4, blockIndependence=False, contentChecksum=False, addContentSize=True):
    return dict(maxBlockSize=maxBlockSize, blockIndependence=blockIndependence, contentChecksum=contentChecksum,
                addContentSize=addContentSize)


def _check_compress(dl, ctx, data, dictionary=None, bc=False, offset=0, **kw):
    kw = _kw(**kw)
    got = _compress_dev(dl, ctx, data, dictionary, kw, bc, offset)
    want = fb._oracle_frame(bytes(data), dictionary, kw, bc)
    assert got == want, (len(data), kw, bc, offset)
    assert got == dl.compressBuffer(data, dictionary, kw["maxBlockSize"], kw["blockIndependence"], kw["contentChecksum"],
                                    kw["addContentSize"], None, bc, ctx=ctx), (len(data), kw, bc)
    return got


# ================================================================================ 1. compress parity
@pytest.mark.parametrize("opts", sorted(GOLDEN_OPTS))
@pytest.mark.parametrize("bc", [False, True])
def test_compress_parity_edge_and_golden_inputs(dl, opts, bc):
    ctx = dl.default_context()
    kw = fb._kw(GOLDEN_OPTS[opts])
    for data in list(edge_corpora().values()) + list(golden_inputs().values()) + [b""]:
        _check_compress(dl, ctx, data, None, bc, **kw)


def test_compress_parity_with_dictionaries(dl):
    from divortio_lz4_b200 import corpus
    ctx = dl.default_context()
    msgs = corpus.jsonmsgs(4, 0, 100).tobytes()
    inputs = [msgs[:4096], msgs[:70000], b"", b"x", msgs[:300000]]
    for dic in (corpus.json_dictionary(44).tobytes(), corpus.jsonmsgs(45, 0, 40).tobytes()[:100000], b"tiny"):
        for indep in (False, True):
            for mbs in (B64, M4):
                for data in inputs:
                    _check_compress(dl, ctx, data, dic, False, maxBlockSize=mbs, blockIndependence=indep, contentChecksum=True)


# ================================================================================ 2. every compress route
def _route_inputs(small):
    """(tag, data, dictionary, kw): the compress routes of frame_body.  small=False at the default thresholds (segment
    engine from 256 KiB), small=True for a context whose segment engine starts at 16 KiB."""
    from divortio_lz4_b200 import corpus
    k = 1 if small else 16
    log = corpus.log(31, 9 * M4 // (16 // k) + 77).tobytes()
    mixed = corpus.mixed(32, 3 * M4 // (16 // k) + 5).tobytes()
    dic = corpus.json_dictionary(33).tobytes()
    yield "short_linked_chain", log[:(12 if small else 200) << 10], None, _kw(B64)
    yield "segments_linked", log, None, _kw(M4)
    yield "segments_linked_64k", mixed, None, _kw(B64, contentChecksum=True)
    yield "segments_independent_4m", log, None, _kw(M4, True)
    yield "segments_independent_256k", mixed, None, _kw(262144, True, True)
    yield "dictionary_block0_then_fresh", mixed, dic, _kw(B64, True)
    yield "dictionary_linked", mixed, dic, _kw(B64, False, True)


def test_every_compress_route_at_real_sizes(dl, ctxs):
    from divortio_lz4_b200 import corpus
    ctx = ctxs["default"]
    for tag, data, dic, kw in _route_inputs(False):
        for bc in (False, True):
            _check_compress(dl, ctx, data, dic, bc, **kw)
    # independent 64 KiB blocks, >= 32 MiB: the host call pipelines them over PCIe, the device call takes launch_compress
    big = corpus.mixed(34, (40 << 20) + 3).tobytes()
    assert len(big) >= 32 << 20
    _check_compress(dl, ctx, big, None, False, maxBlockSize=B64, blockIndependence=True)


def test_every_compress_route_at_small_sizes(dl, ctxs):
    ctx = ctxs["small"]
    for tag, data, dic, kw in _route_inputs(True):
        for bc in (False, True):
            _check_compress(dl, ctx, data, dic, bc, **kw)


# ================================================================================ 3. decompress parity
def _host_decode(dl, ctx, f, dictionary, flags, cap):
    n = C.c_uint64(0)
    out = np.zeros(max(cap, 1) + 64, dtype=np.uint8)
    fa = np.frombuffer(f, dtype=np.uint8) if len(f) else np.zeros(1, dtype=np.uint8)
    d = np.frombuffer(dictionary, dtype=np.uint8) if dictionary else None
    st = dl.api.lib().dlz4_frame_decompress(ctx.handle, fa.ctypes.data, len(f), d.ctypes.data if d is not None else None,
                                            len(dictionary or b""), flags, out.ctypes.data, cap, C.byref(n))
    return st, int(n.value), out[:int(n.value)].tobytes() if st == 0 else b""


def _dev_decode(dl, ctx, f, dictionary, flags, cap, offset=0):
    import torch
    src = _gpu(f if len(f) else b"\0", offset)              # (an empty view's data_ptr() is 0: keep a byte behind it)
    d = _gpu(dictionary, offset) if dictionary else None
    dst = torch.empty(cap + offset, dtype=torch.uint8, device="cuda")[offset:]
    n = C.c_uint64(0)
    st = dl.api.lib().dlz4_frame_decompress_dev(ctx.handle, src.data_ptr(), len(f), _ptr(d), len(dictionary or b""), flags,
                                                _ptr(dst), cap, C.byref(n), C.c_void_p(torch.cuda.current_stream().cuda_stream or 1))
    assert st < 20, st
    return st, int(n.value), dst[:int(n.value)].cpu().numpy().tobytes() if st == 0 else b""


def _valid_frames(dl, kats):
    """Frames of the oracle, liblz4 and the reference's golden vectors."""
    import lz4f
    from divortio_lz4_b200 import corpus
    frames = []
    for name, data in list(golden_inputs().items()) + [("mixed", corpus.mixed(15, 700000).tobytes())]:
        for opts in GOLDEN_OPTS.values():
            frames.append(fb._oracle_frame(data, None, fb._kw(opts), False))
        if lz4f.available():
            for bsid in (4, 7):
                for linked in (False, True):
                    for bc in (False, True):
                        frames.append(lz4f.compress_frame(data, bsid, linked, True, True, bc))
    frames += [bytes.fromhex(k["hex"]) for k in kats["reference_golden"]["decode_frames"]]
    return frames


def _route_frames():
    """Frames whose shape selects each decode route (see frame_decode): with the default thresholds,
    jump decoder  -- a linked frame of >= 256 KiB, and few large independent blocks;
    k_decompress_chain -- a linked frame below 256 KiB;
    strided decode -- full independent 64 KiB blocks; with gap closing -- short inner blocks and no content size (the block
    bound leaves room for n - 1 full blocks); running offsets -- short inner blocks with a content size."""
    rng = np.random.RandomState(90)
    yield "jump_linked", dd.random_frame(rng, 4, True, 6, stored_every=4, cc=True)
    yield "jump_few_large", dd.random_frame(rng, 6, False, 3, large=True, cc=True)
    yield "chain", dd.random_frame(rng, 4, True, 3, full=False)
    yield "strided", dd.random_frame(rng, 4, False, 8, stored_every=3, cc=True)
    yield "strided_gap_closing", dd.random_frame(rng, 4, False, 4, full=False, with_size=False, cc=True)
    fr = dd.random_frame(rng, 4, False, 4, full=False, cc=True)
    assert len(fr.plain) <= 3 * B64                             # no room for three full blocks before the last
    yield "running_offsets", fr
    yield "linked_dict", dd.random_frame(rng, 5, True, 3, dictionary=dd._rb(rng, 70000), cc=True)
    yield "indep_dict", dd.random_frame(rng, 5, False, 3, dictionary=dd._rb(rng, 1000))


def _check_decode(dl, ctx, f, dictionary, flags, tag):
    try:
        cap = int(dl.frame_info(f).max_decoded)
    except dl.LZ4Error:
        cap = 4096
    for c in (cap, max(cap - 1, 0)):
        want = _host_decode(dl, ctx, f, dictionary, flags, c)
        got = _dev_decode(dl, ctx, f, dictionary, flags, c)
        assert got == want, (tag, flags, c, got[:2], want[:2])


@pytest.mark.parametrize("flags", list(range(8)))
def test_decode_parity_valid_frames(dl, ctxs, kats, flags):
    for i, f in enumerate(_valid_frames(dl, kats)):
        for name in ("default", "small"):
            _check_decode(dl, ctxs[name], f, None, flags, (i, name))


@pytest.mark.parametrize("flags", list(range(8)))
def test_decode_parity_every_route(dl, ctxs, flags):
    for tag, fr in _route_frames():
        f = fr.bytes()
        assert dd.frame_model(fr) == fr.plain, tag
        for name, ctx in ctxs.items():
            _check_decode(dl, ctx, f, fr.dictionary, flags, (tag, name))


@pytest.mark.parametrize("flags", list(range(8)))
def test_decode_parity_corrupt_and_error_order_frames(dl, ctxs, flags):
    rng = np.random.RandomState(130 + flags)
    frames, _ = fb._error_frames(dl, rng)
    for i, f in enumerate(frames):
        for name, ctx in ctxs.items():
            _check_decode(dl, ctx, f, None, flags, (i, name))


# ================================================================================ 4. info
_INFO_FIELDS = [f for f, _ in __import__("divortio_lz4_b200").api.FrameInfo._fields_]


def _info_pair(dl, ctx, f):
    import torch
    L = dl.api.lib()
    fa = np.frombuffer(f, dtype=np.uint8) if len(f) else np.zeros(1, dtype=np.uint8)
    hi, di = dl.api.FrameInfo(), dl.api.FrameInfo()
    hs = L.dlz4_frame_info(fa.ctypes.data, len(f), C.byref(hi))
    t = _gpu(f if len(f) else b"\0", 3)
    ds = L.dlz4_frame_info_dev(ctx.handle, t.data_ptr(), len(f), C.byref(di), C.c_void_p(torch.cuda.current_stream().cuda_stream or 1))
    return (hs, [getattr(hi, k) for k in _INFO_FIELDS]), (ds, [getattr(di, k) for k in _INFO_FIELDS])


def test_info_equals_the_host_call(dl, kats):
    ctx = dl.default_context()
    frames = _valid_frames(dl, kats)
    frames += [fb._oracle_frame(b"abc" * 1000, b"dictionary bytes", fb._kw(GOLDEN_OPTS["indep64k_cc"]), True)]
    for f in frames:
        want, got = _info_pair(dl, ctx, f)
        assert got == want
    # every truncation of a header, and of the frame behind it
    for f in frames[::5] + frames[-1:]:
        for k in list(range(0, min(len(f), 24))) + [len(f) - 1, len(f) - 4, len(f) - 5]:
            if k < 0:
                continue
            want, got = _info_pair(dl, ctx, f[:k])
            assert got == want, k


# ================================================================================ 5. caller memory
def test_unaligned_sources_destinations_and_dictionaries(dl):
    from divortio_lz4_b200 import corpus
    ctx = dl.default_context()
    data = corpus.log(40, 700001).tobytes()
    dic = corpus.json_dictionary(41).tobytes()
    for offset in (1, 3, 7):
        for kw in (_kw(), _kw(B64, True, True), _kw(B64, False, True)):
            f = _check_compress(dl, ctx, data, dic, True, offset, **kw)
            assert _dev_decode(dl, ctx, f, dic, 3, len(data), offset) == (0, len(data), data)


def test_frames_and_inputs_that_end_flush_with_their_tensor(dl):
    """The input and the frame end exactly where their tensor ends, and the tensor's size is a multiple of 512 bytes, so it also
    ends at the end of its caching-allocator block (no guarantee of a page end: a read past it would land in a neighbouring
    block, not fault)."""
    import torch
    from divortio_lz4_b200 import corpus, device
    ctx = dl.default_context()
    for n, kw in ((1 << 20, _kw()), (300 * 1024, _kw(B64, True, True)), (4096 * 3, _kw(B64))):
        data = corpus.mixed(42, n).tobytes()
        assert n % 512 == 0
        src = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        f = device.compress_tensor(src, None, **kw)
        want = fb._oracle_frame(data, None, kw, False)
        assert f.cpu().numpy().tobytes() == want
        pad = (-len(want)) % 512
        buf = torch.zeros(len(want) + pad, dtype=torch.uint8, device="cuda")
        buf[pad:] = f
        frame = buf[pad:]
        assert (frame.data_ptr() + frame.numel()) == (buf.data_ptr() + buf.numel())
        assert device.decompress_tensor(frame).cpu().numpy().tobytes() == data


def test_tensor_arguments_are_checked(dl):
    import torch
    from divortio_lz4_b200 import device
    with pytest.raises(ValueError):
        device.compress_tensor(torch.zeros(8, dtype=torch.uint8))
    with pytest.raises(ValueError):
        device.decompress_tensor(torch.zeros(8, dtype=torch.uint8))
    with pytest.raises(ValueError):
        device.compress_tensor(torch.zeros(8, 8, dtype=torch.uint8, device="cuda").t())
    other = types.SimpleNamespace(device=1)                     # a context of another device
    with pytest.raises(ValueError):
        device.compress_tensor(torch.zeros(8, dtype=torch.uint8, device="cuda"), ctx=other)
    with pytest.raises(ValueError):
        device.decompress_tensor(torch.zeros(8, dtype=torch.uint8, device="cuda"), ctx=other)
    # any dtype is its bytes
    x = torch.arange(1000, dtype=torch.float32, device="cuda")
    f = device.compress_tensor(x)
    assert f.cpu().numpy().tobytes() == oracle.compress_buffer(x.cpu().numpy().tobytes())
    with pytest.raises(dl.LZ4Error, match="Unsupported Version 2"):
        device.decompress_tensor(_gpu(bytes.fromhex("04224D18A0400000")))
    with pytest.raises(dl.LZ4Error, match="Content Checksum Error"):
        g = bytearray(oracle.compress_buffer(b"abc" * 100, None, B64, True, True))
        g[-1] ^= 1
        device.decompress_tensor(_gpu(bytes(g)))


# ================================================================================ 6. streams
def test_inputs_written_on_a_side_stream_just_before_the_call(dl):
    import torch
    from divortio_lz4_b200 import corpus, device
    ctx = dl.default_context()
    data = corpus.log(50, (24 << 20) + 11).tobytes()
    want_plain = (np.frombuffer(data, dtype=np.uint8) ^ 0x5A).tobytes()
    want = oracle.compress_buffer(want_plain, None, B64, False, True)
    base = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        x = torch.bitwise_xor(base, 0x5A)                       # queued on s, not finished when the call starts
        f = device.compress_tensor(x, None, B64, False, True)
        g = f.clone()                                           # the frame, written by a torch op just before decoding
        out = device.decompress_tensor(g)
        got_f, got = f.cpu().numpy().tobytes(), out.cpu().numpy().tobytes()
    s.synchronize()
    assert got_f == want
    assert got == want_plain


# ================================================================================ 7. round trip
@pytest.mark.parametrize("kw", [dict(), dict(maxBlockSize=B64, blockIndependence=True)], ids=["default", "indep64k"])
def test_round_trip_256_mib(dl, kw):
    import torch
    from divortio_lz4_b200 import corpus, device
    data = corpus.mixed(60, 256 << 20)
    t = torch.from_numpy(data).cuda()
    f = device.compress_tensor(t, **kw)
    assert f.cpu().numpy().tobytes() == dl.compressBuffer(data, None, kw.get("maxBlockSize", M4), kw.get("blockIndependence", False))
    assert torch.equal(device.decompress_tensor(f), t)
