"""GPU parity, batched frames: compressBuffers / decompressBuffers and the dlz4_frames_*_batch* calls against the oracle and
against the single-frame calls, frame by frame, byte for byte and status for status.  -m gpu."""
import ctypes as C

import numpy as np
import pytest

import oracle
import test_gpu_decode_differential as dd
from conftest import GOLDEN_OPTS, edge_corpora, golden_inputs

pytestmark = pytest.mark.gpu

B64 = 65536


@pytest.fixture(scope="module")
def dl():
    import divortio_lz4_b200 as m
    m.default_context()
    return m


def _kw(opts):
    return dict(maxBlockSize=opts.get("max_block_size", 4194304), blockIndependence=opts.get("block_independence", False),
                contentChecksum=opts.get("content_checksum", False), addContentSize=opts.get("add_content_size", True))


def _oracle_frame(data, dictionary, kw, bc):
    return oracle.compress_buffer(data, dictionary, kw["maxBlockSize"], kw["blockIndependence"], kw["contentChecksum"],
                                  kw["addContentSize"], None, bc)


def _check_compress(dl, inputs, dictionary=None, bc=False, **kw):
    full = dict(maxBlockSize=4194304, blockIndependence=False, contentChecksum=False, addContentSize=True)
    full.update(kw)
    got = dl.compressBuffers(inputs, dictionary, blockChecksum=bc, **full)
    assert len(got) == len(inputs)
    for i, data in enumerate(inputs):
        want = _oracle_frame(bytes(data), dictionary, full, bc)
        assert got[i] == want, (i, len(data), full, bc)
        assert got[i] == dl.compressBuffer(data, dictionary, full["maxBlockSize"], full["blockIndependence"],
                                           full["contentChecksum"], full["addContentSize"], None, bc), (i, len(data))
    return got


# ================================================================================ compress parity
@pytest.mark.parametrize("opts", sorted(GOLDEN_OPTS))
@pytest.mark.parametrize("bc", [False, True])
def test_compress_parity_edge_and_golden_inputs(dl, opts, bc):
    inputs = list(edge_corpora().values()) + list(golden_inputs().values()) + [b"", b""]
    frames = _check_compress(dl, inputs, None, bc, **_kw(GOLDEN_OPTS[opts]))
    assert dl.decompressBuffers(frames, None, True, True) == [bytes(x) for x in inputs]


def test_compress_parity_with_dictionaries(dl):
    from divortio_lz4_b200 import corpus
    msgs = corpus.jsonmsgs(4, 0, 100).tobytes()
    inputs = [msgs[i * 4096:(i + 1) * 4096] for i in range(20)] + [msgs, msgs[:70000], b"", b"x", msgs[:300000]]
    for dic in (corpus.json_dictionary(44).tobytes(), corpus.jsonmsgs(45, 0, 40).tobytes()[:100000], b"tiny"):
        for indep in (False, True):
            for mbs in (B64, 4194304):
                frames = _check_compress(dl, inputs, dic, False, maxBlockSize=mbs, blockIndependence=indep, contentChecksum=True)
                assert dl.decompressBuffers(frames, dic) == inputs, (len(dic), indep, mbs)


def test_compress_parity_around_block_boundaries(dl):
    from divortio_lz4_b200 import corpus
    base = corpus.mixed(7, 3 * B64 + 5).tobytes()
    inputs = [base[:B64 - 1], base[:B64], base[:B64 + 1], base]
    for indep in (False, True):
        for bc in (False, True):
            frames = _check_compress(dl, inputs, None, bc, maxBlockSize=B64, blockIndependence=indep, contentChecksum=bc)
            assert dl.decompressBuffers(frames, None, True, True) == inputs


# ================================================================================ shapes
def test_one_and_seven_frames(dl):
    from divortio_lz4_b200 import corpus
    data = corpus.log(3, 200000).tobytes()
    _check_compress(dl, [data])
    _check_compress(dl, [data[i * 1000:(i + 1) * 27000] for i in range(7)], None, True, maxBlockSize=B64, contentChecksum=True)


def test_hundred_thousand_messages_behind_a_dictionary(dl):
    from divortio_lz4_b200 import corpus
    n = 100000
    raw = corpus.jsonmsgs(11, 0, n).tobytes()
    dic = corpus.json_dictionary(11).tobytes()
    msgs = [raw[i * 4096:(i + 1) * 4096] for i in range(n)]
    frames = dl.compressBuffers(msgs, dic, contentChecksum=True)
    rng = np.random.RandomState(12)
    for i in rng.choice(n, 2000, replace=False):
        assert frames[i] == oracle.compress_buffer(msgs[i], dic, 4194304, False, True), i
    assert dl.decompressBuffers(frames, dic) == msgs


def test_mixed_sizes_up_to_nine_mib(dl):
    from divortio_lz4_b200 import corpus
    rng = np.random.RandomState(13)
    sizes = [0, 1, 17, 4096, 65535, 65536, 65537, 300000, 1 << 20, (4 << 20) + 3, 9 << 20] + list(rng.randint(0, 200000, 40))
    data = corpus.mixed(14, sum(sizes)).tobytes()
    inputs, p = [], 0
    for s in sizes:
        inputs.append(data[p:p + s])
        p += s
    for indep in (False, True):
        frames = _check_compress(dl, inputs, None, True, maxBlockSize=B64 if indep else 4194304, blockIndependence=indep,
                                 contentChecksum=True)
        assert dl.decompressBuffers(frames, None, True, True) == inputs


# ================================================================================ decode parity
def test_decode_frames_of_every_writer_in_one_batch(dl, kats):
    import lz4f
    from divortio_lz4_b200 import corpus
    frames, plains = [], []
    for name, data in list(golden_inputs().items()) + [("mixed", corpus.mixed(15, 700000).tobytes())]:
        for opts in GOLDEN_OPTS.values():
            kw = _kw(opts)
            frames.append(_oracle_frame(data, None, kw, False))
            plains.append(data)
        if lz4f.available():
            for bsid in (4, 7):
                for linked in (False, True):
                    for size in (False, True):
                        for bc in (False, True):
                            frames.append(lz4f.compress_frame(data, bsid, linked, True, size, bc))
                            plains.append(data)
    for k in kats["reference_golden"]["decode_frames"]:
        frames.append(bytes.fromhex(k["hex"]))
        plains.append(k["text"].encode())
    assert dl.decompressBuffers(frames, None, True, True) == plains


# ================================================================================ errors: every frame as the single call sees it
def _single(dl, ctx, f, dictionary, flags, cap):
    n = C.c_uint64(0)
    out = np.zeros(max(cap, 1) + 64, dtype=np.uint8)
    fa = np.frombuffer(f, dtype=np.uint8) if len(f) else np.zeros(1, dtype=np.uint8)
    d = np.frombuffer(dictionary, dtype=np.uint8) if dictionary else None
    st = dl.api.lib().dlz4_frame_decompress(ctx.handle, fa.ctypes.data, len(f), d.ctypes.data if d is not None else None,
                                            len(dictionary or b""), flags, out.ctypes.data, cap, C.byref(n))
    return (st, int(n.value) if st == 0 else 0, out[:int(n.value)].tobytes() if st == 0 else b"")


def _batch(dl, ctx, frames, dictionary, flags, caps):
    src, off, lens = dl.api._concat(frames)
    n = len(frames)
    caps = np.array(caps, dtype=np.uint64)
    doff = np.zeros(n, dtype=np.uint64)
    doff[1:] = np.cumsum(caps + 16)[:-1]
    dst = np.zeros(int((caps + 16).sum()) + 16, dtype=np.uint8)
    out_len = np.zeros(n, dtype=np.uint64)
    status = np.zeros(n, dtype=np.uint8)
    d = np.frombuffer(dictionary, dtype=np.uint8) if dictionary else None
    st = dl.api.lib().dlz4_frames_decompress_batch(ctx.handle, src.ctypes.data, src.size, off.ctypes.data, lens.ctypes.data, n,
                                                   d.ctypes.data if d is not None else None, len(dictionary or b""), flags,
                                                   dst.ctypes.data, dst.size, doff.ctypes.data, caps.ctypes.data,
                                                   out_len.ctypes.data, status.ctypes.data)
    assert st < 20, st
    first = next((int(s) for s in status if s), 0)
    assert st == first
    return [(int(status[i]), int(out_len[i]), dst[int(doff[i]):int(doff[i]) + int(out_len[i])].tobytes()) for i in range(n)]


def _caps(dl, frames):
    caps = []
    for f in frames:
        try:
            caps.append(int(dl.frame_info(f).max_decoded))
        except dl.LZ4Error:
            caps.append(4096)
    return caps


def _error_frames(dl, rng):
    """Good frames mixed with corrupt ones: mutated blocks, the error-order cases, header and table damage, flipped checksums."""
    from divortio_lz4_b200 import corpus
    good, bad = [], []
    plain = corpus.log(21, 300000).tobytes()
    for indep in (False, True):
        for mbs in (B64, 4194304):
            good.append(dl.compressBuffer(plain, None, mbs, indep, True, True, None, True))
    good.append(dl.compressBuffer(b"", None, B64, True, True))
    for bd, linked, nb, kw in [(4, True, 3, {}), (4, False, 3, dict(cc=True)), (5, True, 2, dict(stored_every=2)),
                               (4, False, 2, dict(with_size=False, cc=True))]:
        fr = dd.random_frame(rng, bd, linked, nb, **kw)
        good.append(fr.bytes())
        for k, (payload, stored) in enumerate(fr.blocks):
            if stored:
                continue
            for m in list(dd.mutations(rng, payload, False))[:6]:
                blocks = list(fr.blocks)
                blocks[k] = (m, False)
                bad.append(fr.with_blocks(blocks).bytes())
    for build in (dd.case_a, dd.case_a_later_block, dd.case_b, dd.case_c):
        bad.append(build(rng).bytes())
    g = good[0]
    bad += [b"\x00\x01\x02\x03\x04\x05\x06\x07", bytes.fromhex("04224D18A0400000"), b"\x04\x22\x4d", g[:7], g[:len(g) // 2],
            g[:-1], g[:-6]]
    flip = bytearray(g)
    flip[-1] ^= 0xFF                                                # content checksum
    bad.append(bytes(flip))
    flip = bytearray(good[1])
    flip[40] ^= 0x01                                                # inside block 0's payload: block checksum
    bad.append(bytes(flip))
    hc = bytearray(g)
    hc[14] ^= 0x55                                                  # header checksum byte (content size present, no dict)
    bad.append(bytes(hc))
    frames = []
    for i in range(max(len(good), len(bad))):                       # interleaved
        if i < len(good):
            frames.append(good[i])
        if i < len(bad):
            frames.append(bad[i])
    return frames, good


@pytest.mark.parametrize("flags", [0, 1, 2, 3, 4, 7])
def test_errors_match_the_single_frame_call(dl, flags):
    ctx = dl.default_context()
    rng = np.random.RandomState(30 + flags)
    frames, good = _error_frames(dl, rng)
    caps = _caps(dl, frames)
    got = _batch(dl, ctx, frames, None, flags, caps)
    for i, f in enumerate(frames):
        want = _single(dl, ctx, f, None, flags, caps[i])
        assert got[i] == want, (i, flags, got[i][:2], want[:2])
    assert sum(1 for g in got if g[0] == 0) >= len(good)
    # one byte too small: the decoder's OUTPUT_TOO_SMALL, as the single call reports it
    tight = [max(c - 1, 0) for c in caps]
    got = _batch(dl, ctx, frames, None, flags, tight)
    for i, f in enumerate(frames):
        assert got[i] == _single(dl, ctx, f, None, flags, tight[i]), (i, flags)


def test_errors_raise_or_return(dl):
    from divortio_lz4_b200 import corpus
    data = corpus.log(22, 5000).tobytes()
    f = dl.compressBuffer(data, None, B64, False, True)
    frames = [f, bytes.fromhex("04224D18A0400000"), f]
    with pytest.raises(dl.LZ4Error, match="Unsupported Version 2"):
        dl.decompressBuffers(frames)
    got = dl.decompressBuffers(frames, errors="return")
    assert got[0] == data and got[2] == data
    assert isinstance(got[1], dl.LZ4Error) and str(got[1]) == "LZ4: Unsupported Version 2" and got[1].status == 6
    with pytest.raises(dl.LZ4Error, match="Invalid Magic Number"):
        dl.decompressBuffers([f, b"\x00" * 12])


def test_dictionary_frames_decode_with_the_dictionary(dl):
    from divortio_lz4_b200 import corpus
    dic = corpus.json_dictionary(44).tobytes()
    raw = corpus.jsonmsgs(5, 0, 64).tobytes()
    msgs = [raw[i * 4096:(i + 1) * 4096] for i in range(64)] + [raw]
    ctx = dl.default_context()
    for indep in (False, True):
        frames = dl.compressBuffers(msgs, dic, B64, indep, True)
        caps = _caps(dl, frames)
        got = _batch(dl, ctx, frames, dic, 1, caps)
        assert [g[2] for g in got] == msgs
        for i in (0, 63, 64):
            assert got[i] == _single(dl, ctx, frames[i], dic, 1, caps[i])


# ================================================================================ device forms
def test_device_forms_on_a_side_stream_equal_the_host_forms(dl):
    import torch
    from divortio_lz4_b200 import corpus, device
    ctx = dl.default_context()
    raw = corpus.jsonmsgs(6, 0, 300).tobytes()
    dic = corpus.json_dictionary(6).tobytes()
    msgs = [raw[i * 4096:i * 4096 + 100 + 13 * i] for i in range(300)] + [raw, b""]
    opts_kw = dict(maxBlockSize=B64, blockIndependence=False, contentChecksum=True, addContentSize=True, blockChecksum=True)
    want = dl.compressBuffers(msgs, dic, **opts_kw)
    src, off, lens = dl.api._concat(msgs)
    dev = torch.device("cuda")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        t_src = torch.from_numpy(src).to(dev)
        t_off = torch.from_numpy(off.astype(np.int64)).to(dev)
        t_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
        t_dic = torch.frombuffer(bytearray(dic), dtype=torch.uint8).to(dev)
        cap = int((19 + lens + (lens // 65536 + 1) * 8 + 8 + 64).sum())
        t_dst = torch.zeros(cap, dtype=torch.uint8, device=dev)
        t_fo = torch.zeros(len(msgs) + 1, dtype=torch.int64, device=dev)
        device.frames_compress_batch_dev(ctx, t_src, t_off, t_len, int(lens.max()), t_dst, t_fo, dl.api.frame_opts(**opts_kw), t_dic)
        fo = t_fo.cpu().numpy()
        dst = t_dst.cpu().numpy()
    s.synchronize()
    got = [dst[fo[i]:fo[i + 1]].tobytes() for i in range(len(msgs))]
    assert got == want
    fsrc, foff, flen = dl.api._concat(want)
    with torch.cuda.stream(s):
        t_fs = torch.from_numpy(fsrc).to(dev)
        t_foff = torch.from_numpy(foff.astype(np.int64)).to(dev)
        t_flen = torch.from_numpy(flen.astype(np.int64)).to(dev)
        t_md = torch.zeros(len(want), dtype=torch.int64, device=dev)
        t_ist = torch.zeros(len(want), dtype=torch.uint8, device=dev)
        device.frames_batch_info_dev(ctx, t_fs, t_foff, t_flen, t_md, t_ist)
        md = t_md.cpu().numpy().astype(np.uint64)
        doff = np.zeros(len(want), dtype=np.uint64)
        doff[1:] = np.cumsum(md)[:-1]
        t_out = torch.zeros(int(md.sum()) + 16, dtype=torch.uint8, device=dev)
        t_doff = torch.from_numpy(doff.astype(np.int64)).to(dev)
        t_olen = torch.zeros(len(want), dtype=torch.int64, device=dev)
        t_st = torch.full((len(want),), 99, dtype=torch.uint8, device=dev)
        device.frames_decompress_batch_dev(ctx, t_fs, t_foff, t_flen, t_out, t_doff, t_md, t_olen, t_st, t_dic, flags=3)
        st, olen, out = t_st.cpu().numpy(), t_olen.cpu().numpy(), t_out.cpu().numpy()
        ist = t_ist.cpu().numpy()
    s.synchronize()
    assert not ist.any() and not st.any()
    assert [out[int(doff[i]):int(doff[i]) + int(olen[i])].tobytes() for i in range(len(want))] == msgs
    assert dl.decompressBuffers(want, dic, True, True) == msgs
