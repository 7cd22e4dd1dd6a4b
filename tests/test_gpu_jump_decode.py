"""GPU parity, jump decoder (k_jd_*): linked-block frames (bufferDecompress.js:153) and frames of few large blocks are decoded
by a token scan plus pointer doubling instead of one warp per dependent stream.  Output must equal the oracle's / the input,
errors must be the reference's.  -m gpu."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dl():
    import divortio_lz4_b200 as m
    m.default_context()
    return m


def _corpora(n):
    from divortio_lz4_b200 import corpus
    return {
        "log": corpus.log(31, n).tobytes(),
        "mixed": corpus.mixed(32, n).tobytes(),
        "zero": bytes(n),                                            # one copy chain as deep as the block
        "rand": corpus.rand(33, n).tobytes(),                        # stored blocks
        "bench": corpus.benchjson(n).tobytes(),                      # period 219
        "periods": (b"".join(bytes((j * 7 + p) & 0xFF for j in range(p)) * (60000 // p + 3) for p in range(1, 41)) * 2)[:n],
        "2sym": np.random.RandomState(5).choice(np.frombuffer(b"ab", dtype=np.uint8), n).tobytes(),
    }


@pytest.mark.parametrize("bs", [65536, 262144, 1048576, 4194304])
def test_linked_frames_from_the_oracle(dl, bs):
    n = 9 * 1024 * 1024 + 4321
    for name, data in _corpora(n).items():
        f = oracle.compress_buffer(data, None, bs, False, True, True)
        assert dl.decompressBuffer(f) == data, name


@pytest.mark.parametrize("bs", [262144, 4194304])
def test_few_large_independent_blocks(dl, bs):
    n = 13 * 1024 * 1024 + 99
    for name, data in _corpora(n).items():
        f = oracle.compress_buffer(data, None, bs, True, True, True, None, True)
        assert dl.decompressBuffer(f, None, True, True) == data, name


def test_linked_frame_with_dictionary(dl):
    from divortio_lz4_b200 import corpus
    data = corpus.jsonmsgs(4, 0, 700).tobytes()
    for dic in (corpus.json_dictionary(44).tobytes(), corpus.jsonmsgs(45, 0, 40).tobytes()[:100000], b"tiny"):
        for bs in (65536, 1048576):
            f = oracle.compress_buffer(data, dic, bs, False, True)
            assert dl.decompressBuffer(f, dic) == data
            with pytest.raises(dl.LZ4Error):                         # without the dictionary: offsets reach before the output
                if dl.decompressBuffer(f, None, False) == data:
                    raise dl.LZ4Error(0, "dictionary was not needed")   # tiny dictionaries may never be referenced


def test_liblz4_linked_frames_with_and_without_content_size(dl):
    import lz4f
    if not lz4f.available():
        pytest.skip("liblz4 not present")
    n = 11 * 1024 * 1024 + 5
    for name, data in _corpora(n).items():
        for bsid in (4, 7):
            for size in (False, True):
                f = lz4f.compress_frame(data, bsid, True, True, size, True)
                assert dl.decompressBuffer(f, None, True, True) == data, (name, bsid, size)


def test_corrupt_linked_frames_raise_the_reference_errors(dl):
    from divortio_lz4_b200 import corpus
    data = corpus.log(41, 3 * 1024 * 1024).tobytes()
    f = bytearray(oracle.compress_buffer(data, None, 1048576, False, False, True))
    # zero offset in the middle of block 1
    g = bytearray(f)
    pos = len(g) // 2
    for k in range(pos, pos + 4000):
        g[k] = 0
    with pytest.raises(oracle.OracleError) as want:
        oracle.decompress_buffer(bytes(g))
    with pytest.raises(dl.LZ4Error) as ei:
        dl.decompressBuffer(bytes(g))
    assert ei.value.status == -want.value.code and str(ei.value) == str(want.value)
    # truncated frame
    with pytest.raises(dl.LZ4Error):
        dl.decompressBuffer(bytes(f[: len(f) // 3]))
    # declared content size too small -> Output Buffer Too Small, like the reference's fixed-size allocation
    h = bytearray(f)
    h[6:14] = (1000).to_bytes(8, "little")
    h[14] = (oracle.xxh32(bytes(h[4:14])) >> 8) & 0xFF
    with pytest.raises(dl.LZ4Error, match="Output Buffer Too Small"):
        dl.decompressBuffer(bytes(h))


def test_jump_and_chain_decoders_agree_on_a_short_linked_frame(dl):
    """Frames under 256 KiB take the single-warp chain kernel; a second context with the threshold at 0 takes the jump path."""
    import os
    from divortio_lz4_b200 import corpus
    data = corpus.log(51, 200000).tobytes()
    f = oracle.compress_buffer(data, None, 65536, False, True)
    assert dl.decompressBuffer(f) == data
    os.environ["DLZ4_JUMP_MIN_KIB"] = "0"
    try:
        ctx = dl.Context(0)
        assert dl.decompressBuffer(f, None, True, False, ctx=ctx) == data
        for k in (0, 1, 13, 70000):
            d2 = corpus.log(52, k).tobytes()
            assert dl.decompressBuffer(oracle.compress_buffer(d2, None, 65536, False, True), None, True, False, ctx=ctx) == d2
    finally:
        del os.environ["DLZ4_JUMP_MIN_KIB"]
