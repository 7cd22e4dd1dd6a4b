"""GPU parity, frame layer: compressBuffer / decompressBuffer through the C ABI vs the oracle, byte for byte.  -m gpu."""
import numpy as np
import pytest

import oracle
from conftest import GOLDEN_OPTS, edge_corpora, golden_inputs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dl():
    import divortio_lz4_b200 as m
    m.default_context()
    return m


def _gpu_frame(dl, data, dictionary=None, max_block_size=4194304, block_independence=False, content_checksum=False,
               add_content_size=True, block_checksum=False):
    return dl.compressBuffer(data, dictionary, max_block_size, block_independence, content_checksum, add_content_size, None,
                             block_checksum)


def test_golden_fixture_frames(dl, kats):
    ins = golden_inputs()
    for rec in kats["frames"]:
        f = _gpu_frame(dl, ins[rec["input"]], None, **GOLDEN_OPTS[rec["opts"]])
        assert len(f) == rec["len"] and oracle.xxh32(f) == rec["xxh32"], rec
        if "hex" in rec:
            assert f.hex() == rec["hex"]
        assert dl.decompressBuffer(f) == ins[rec["input"]]


def test_reference_golden_decode_frames(dl, kats):
    for k in kats["reference_golden"]["decode_frames"]:
        assert dl.decompressBuffer(bytes.fromhex(k["hex"])) == k["text"].encode()


def test_dictionary_frames(dl, kats):
    for rec in kats["dictionary"]:
        data = bytes.fromhex(rec["input_hex"])
        d = bytes.fromhex(rec["dict_hex"]) if "dict_hex" in rec else data[:rec["dict_len"]]
        if rec["name"] == "D1":
            f = _gpu_frame(dl, data, d)
        elif rec["name"].endswith("indep_cc"):
            f = _gpu_frame(dl, data, d, 65536, True, True, True)
        else:
            f = _gpu_frame(dl, data, d, 65536, False, False, True)
        assert f.hex() == rec["hex"], rec["name"]
        assert dl.decompressBuffer(f, d) == data


@pytest.mark.parametrize("indep", [False, True])
@pytest.mark.parametrize("cc", [False, True])
@pytest.mark.parametrize("bc", [False, True])
def test_edge_corpora_all_flag_combinations(dl, indep, cc, bc):
    for name, data in edge_corpora().items():
        f = _gpu_frame(dl, data, None, 65536, indep, cc, True, bc)
        assert f == oracle.compress_buffer(data, None, 65536, indep, cc, True, None, bc), name
        assert dl.decompressBuffer(f, None, True, True) == data, name


@pytest.mark.parametrize("bs", [65536, 262144, 1048576, 4194304])
@pytest.mark.parametrize("indep", [False, True])
def test_multiblock_mixed_corpus(dl, bs, indep):
    from divortio_lz4_b200 import corpus
    n = 9 * 1024 * 1024 + 4321
    data = corpus.mixed(bs + indep, n)
    f = _gpu_frame(dl, data, None, bs, indep, True, True, True)
    want = oracle.compress_buffer(data, None, bs, indep, True, True, None, True)
    assert len(f) == len(want) and f == want
    assert dl.decompressBuffer(f, None, True, True) == data.tobytes()


def test_dictionary_multiblock_both_modes(dl):
    from divortio_lz4_b200 import corpus
    data = corpus.jsonmsgs(4, 0, 100).tobytes()                    # 400 KiB
    for dic in (corpus.json_dictionary(44).tobytes(), corpus.jsonmsgs(45, 0, 40).tobytes()[:100000], b"tiny"):
        for indep in (False, True):
            f = _gpu_frame(dl, data, dic, 65536, indep, True)
            assert f == oracle.compress_buffer(data, dic, 65536, indep, True), (len(dic), indep)
            assert dl.decompressBuffer(f, dic) == data


def test_block_size_quantisation_and_output_buffer(dl):
    data = bytes(range(256)) * 1200                                   # 307200 bytes
    for mbs in (0, 1, 65536, 65537, 262144, 262145, 1048576, 1048577, 4194304, 10 ** 9):
        assert _gpu_frame(dl, data, None, mbs, True) == oracle.compress_buffer(data, None, mbs, True), mbs
    out = np.zeros(dl.frame_bound(len(data)), dtype=np.uint8)
    view = dl.compressBuffer(data, None, 65536, True, False, True, out)
    assert view.base is out or view.base is out.base
    assert view.tobytes() == oracle.compress_buffer(data, None, 65536, True)
    # undersized outputBuffer: silently truncated, like typed-array stores past the end
    small = np.zeros(100, dtype=np.uint8)
    view = dl.compressBuffer(data, None, 65536, True, False, True, small)
    assert view.tobytes() == oracle.compress_buffer(data, None, 65536, True)[:100]


def test_decompress_errors(dl):
    d = b"some payload that repeats, some payload that repeats" * 20
    f = bytearray(_gpu_frame(dl, d, None, 4194304, False, True))
    f[-1] ^= 0xFF
    with pytest.raises(dl.LZ4Error, match="Content Checksum Error"):
        dl.decompressBuffer(bytes(f))
    assert dl.decompressBuffer(bytes(f), None, False) == d
    with pytest.raises(dl.LZ4Error, match="Invalid Magic Number"):
        dl.decompressBuffer(b"\x00\x01\x02\x03\x04\x05\x06\x07")
    with pytest.raises(dl.LZ4Error, match="Unsupported Version 2"):
        dl.decompressBuffer(bytes.fromhex("04224D18A0400000"))
    g = bytearray(_gpu_frame(dl, d * 40, None, 65536, True, False, True, True))
    g[40] ^= 0x01
    with pytest.raises(dl.LZ4Error):
        dl.decompressBuffer(bytes(g), None, True, True)


def test_accepts_liblz4_cli_equivalent_frames(dl):
    import lz4f
    if not lz4f.available():
        pytest.skip("liblz4 not present")
    from divortio_lz4_b200 import corpus
    data = corpus.mixed(12, 5 * 1024 * 1024 + 999).tobytes()
    for bsid in (4, 5, 6, 7):
        for linked in (False, True):
            for size in (False, True):
                for bc in (False, True):
                    f = lz4f.compress_frame(data, bsid, linked, True, size, bc)
                    assert dl.decompressBuffer(f, None, True, True) == data, (bsid, linked, size, bc)
    assert dl.decompressBuffer(lz4f.compress_frame(b"", 4)) == b""


def test_gpu_frames_decode_in_liblz4(dl):
    import lz4f
    if not lz4f.available():
        pytest.skip("liblz4 not present")
    from divortio_lz4_b200 import corpus
    data = corpus.mixed(13, 3 * 1024 * 1024 + 17).tobytes()
    for bs in (65536, 4194304):
        for indep in (False, True):
            f = _gpu_frame(dl, data, None, bs, indep, True, True, True)
            assert lz4f.decompress_frame(f, len(data)) == data


def test_concatenated_and_skippable_frames(dl):
    """SURVEY 8 f3: `cat a.lz4 b.lz4`, skippable frames between them (LZ4 frame spec); decompressBuffer itself keeps the reference's
    one-frame behaviour (bufferDecompress.js stops at the first EndMark)."""
    import struct
    from divortio_lz4_b200 import corpus
    a = corpus.log(61, 300000).tobytes()
    b = corpus.mixed(62, 700001).tobytes()
    c = b""
    fa = oracle.compress_buffer(a, None, 65536, True, True, True)
    fb = oracle.compress_buffer(b, None, 4194304, False, True, False)          # linked, no content size -> jump decoder
    fc = oracle.compress_buffer(c)
    skip = struct.pack("<II", 0x184D2A53, 11) + b"hello world"
    cat = skip + fa + skip + skip + fb + fc + skip
    out, count = dl.decompressFrames(cat, None, True)
    assert count == 3 and out == a + b + c
    assert dl.decompressBuffer(fa + fb) == a                                     # reference behaviour: first frame only
    import lz4f
    if lz4f.available():
        cat2 = lz4f.compress_frame(a, 4, True, True, False, True) + lz4f.compress_frame(b, 7, False, True, True, False)
        out2, count2 = dl.decompressFrames(cat2, None, True, True)
        assert count2 == 2 and out2 == a + b
    with pytest.raises(dl.LZ4Error, match="Invalid Magic"):
        dl.decompressFrames(fa + b"\x01\x02\x03\x04\x05")
    bad = bytearray(fa + fb)
    bad[-1] ^= 0x55                                                              # second frame's content checksum
    with pytest.raises(dl.LZ4Error, match="Content Checksum"):
        dl.decompressFrames(bytes(bad))


def test_large_independent_frame_takes_the_pipelined_path(dl):
    """Frames of >= 32 MiB in independent 64 KiB blocks go through the chunked host pipeline (frame body packed per chunk)."""
    from divortio_lz4_b200 import corpus
    from test_gpu_decode_differential import frame_model, parse_frame
    n = 40 * 1024 * 1024 + 1234
    data = corpus.mixed(71, n)
    for bc in (False, True):
        for size in (True, False):
            f = dl.compressBuffer(data, None, 65536, True, False, size, None, bc)
            want = oracle.compress_buffer(data, None, 65536, True, False, size, None, bc)
            assert len(f) == len(want) and f == want, (bc, size)
    assert dl.decompressBuffer(f, None, True, True) == data.tobytes()
    # decode side of the pipeline (declared size, no block-checksum verification asked): content-size frames, checksummed or not
    for cc in (False, True):
        g = oracle.compress_buffer(data, None, 65536, True, cc, True)
        assert dl.decompressBuffer(g) == data.tobytes()
        bad = bytearray(g)
        bad[len(bad) // 2] ^= 0xFF                                   # somewhere inside a block: the general path names the error
        # the reference's result, with an independent block's history the dictionary only (test_gpu_decode_differential)
        want = frame_model(parse_frame(bytes(bad)), verify_checksum=False)
        if isinstance(want, int):
            with pytest.raises(dl.LZ4Error) as ei:
                dl.decompressBuffer(bytes(bad), None, False)
            assert ei.value.status == want and str(ei.value) == oracle.MESSAGES[-want]
        else:
            assert dl.decompressBuffer(bytes(bad), None, False) == want
        if cc:
            tail = bytearray(g); tail[-2] ^= 1
            with pytest.raises(dl.LZ4Error, match="Content Checksum Error"):
                dl.decompressBuffer(bytes(tail))


def _flushed_frame(pieces, bd, with_size, stored_first=False):
    """A spec-valid independent-block frame whose inner blocks are SHORT (what LZ4F_flush-style writers and a stream's
    update() produce): header by hand, every piece one block compressed by the oracle (stored when that is not smaller)."""
    import struct
    from divortio_lz4_b200 import sharded
    total = sum(len(p) for p in pieces)
    flg = 0x40 | 0x20 | (0x08 if with_size else 0)
    desc = bytes([flg, bd << 4]) + (struct.pack("<Q", total) if with_size else b"")
    out = bytearray(struct.pack("<I", 0x184D2204) + desc + bytes([(oracle.xxh32(desc) >> 8) & 0xFF]))
    for k, p in enumerate(pieces):
        c = oracle.compress_block_bytes(np.frombuffer(p, dtype=np.uint8))
        if (stored_first and k == 0) or len(c) >= len(p):
            out += struct.pack("<I", len(p) | 0x80000000) + p
        else:
            out += struct.pack("<I", len(c)) + c
    out += struct.pack("<I", 0)
    return bytes(out), b"".join(pieces)


@pytest.mark.parametrize("with_size", [False, True])
def test_short_inner_blocks_decode_at_running_offsets(dl, with_size):
    """ADVICE r1 (medium): content_size = 3B with blocks [B/2, B, B, B/2] must decode (the reference decodes sequentially at
    resultPos, bufferDecompress.js:133-192); so must small blocks under a large blockMaxSize and a stored short first block."""
    from divortio_lz4_b200 import corpus
    B = 65536
    text = corpus.log(11, 3 * B).tobytes()
    cases = [
        ([text[:B // 2], text[B // 2:B // 2 + B], text[B // 2 + B:B // 2 + 2 * B], text[B // 2 + 2 * B:]], 4, False),
        ([text[i:i + 1000] for i in range(0, 40000, 1000)], 7, False),            # 40 small blocks, blockMaxSize 4 MiB
        ([text[:100], text[100:100 + B], text[100 + B:2 * B]], 4, True),          # stored short block first
        ([corpus.rand(5, 3000).tobytes(), text[:B], corpus.zero(70).tobytes(), text[B:B + 5]], 4, False),
    ]
    for pieces, bd, stored_first in cases:
        frame, plain = _flushed_frame(pieces, bd, with_size, stored_first)
        assert oracle.decompress_buffer(frame) == plain
        assert dl.decompressBuffer(frame) == plain
        info = dl.frame_info(frame)
        assert info.nblocks == len(pieces)


@pytest.mark.parametrize("seed", [11, 12])
def test_frames_fuzz_random_structured_inputs(dl, seed):
    """Differential fuzz of the frame paths (segment-parallel linked chains, large independent blocks, 64 KiB batches, dictionary
    warm-up, jump decoder) on random structured inputs: frame bytes == oracle for random options, and back."""
    from test_gpu_blocks import _fuzz_block
    import lz4f
    rng = np.random.RandomState(seed)
    for case in range(5):
        n = int(rng.randint(300000, 6000000))
        data = np.frombuffer(_fuzz_block(rng, n), dtype=np.uint8)
        bs = int(rng.choice([65536, 262144, 1048576, 4194304]))
        indep, cc, bc = bool(rng.randint(0, 2)), bool(rng.randint(0, 2)), bool(rng.randint(0, 2))
        dic = np.frombuffer(_fuzz_block(rng, int(rng.randint(100, 90000))), dtype=np.uint8) if rng.randint(0, 3) == 0 else None
        want = oracle.compress_buffer(data, dic, bs, indep, cc, True, None, bc)
        got = dl.compressBuffer(data, dic, bs, indep, cc, True, None, bc)
        assert got == want, (seed, case, n, bs, indep, cc, bc, dic is not None)
        assert dl.decompressBuffer(got, dic, True, bc) == data.tobytes(), (seed, case)
        if lz4f.available() and dic is None:
            assert lz4f.decompress_frame(got, n) == data.tobytes(), (seed, case)
