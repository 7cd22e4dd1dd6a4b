"""GPU parity of the producer/walker match finder (k_parse_pw) at batch sizes that fill its CTAs in different ways: one block,
fewer and more blocks than SMs, every team of every CTA busy plus one block from the work queue; blocks too short for a ring
window (< 112 bytes) and blocks of exactly 64 KiB; two batches in a row on a fresh context (the kernel allocates and frees tensor
memory in every launch).  Compressed bytes are compared with the oracle block by block.  Run with -m gpu."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

TEAMS_PER_CTA = 7


@pytest.fixture(scope="module")
def dl():
    import divortio_lz4_b200 as m
    m.default_context()          # raises if the CUDA library or device is missing: no silent fallback
    return m


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _batch(seed, lens):
    """Blocks of the given lengths cut back to back from a mixed corpus (log text, JSON, zero runs, noise)."""
    from divortio_lz4_b200 import corpus
    lens = [int(x) for x in lens]
    data = corpus.mixed(seed, sum(lens) + 64)
    off = np.concatenate([[0], np.cumsum(lens[:-1])]).astype(np.uint64)
    return data, off, np.array(lens, dtype=np.uint32)


def _assert_like_oracle(dl, data, off, ln, ctx=None):
    dst, doff, clen = dl.compress_blocks(data, off, ln, ctx=ctx)
    odst, odoff, oclen = oracle.compress_blocks(data, off, ln)
    bad = [i for i in range(len(ln)) if clen[i] != oclen[i] or not np.array_equal(dst[int(doff[i]):int(doff[i]) + int(clen[i])],
                                                                                   odst[int(odoff[i]):int(odoff[i]) + int(oclen[i])])]
    assert not bad, ("blocks differ from the oracle", [(i, int(ln[i])) for i in bad[:10]])


def _lens(rng, n):
    # every length class: short, around the window sizes, up to 64 KiB
    return np.where(rng.randint(0, 4, size=n) == 0, 65536, rng.randint(0, 65537, size=n))


@pytest.mark.parametrize("nblocks", ["1", "7", "8", "sm*7+1"])
def test_batch_sizes_bit_exact(dl, nblocks):
    n = _sm_count() * TEAMS_PER_CTA + 1 if nblocks == "sm*7+1" else int(nblocks)
    rng = np.random.RandomState(7000 + n)
    data, off, ln = _batch(5, _lens(rng, n))
    _assert_like_oracle(dl, data, off, ln)


def test_blocks_without_ring_windows(dl):
    """Blocks below 112 bytes have no producer windows: the walker parses them alone, its producers idle."""
    rng = np.random.RandomState(7100)
    lens = list(range(0, 112)) + [int(x) for x in rng.randint(0, 112, size=_sm_count() * TEAMS_PER_CTA)] + [112, 113]
    data, off, ln = _batch(6, lens)
    _assert_like_oracle(dl, data, off, ln)


def test_full_64k_blocks(dl):
    data, off, ln = _batch(7, [65536] * (_sm_count() * TEAMS_PER_CTA + 1))
    _assert_like_oracle(dl, data, off, ln)


def test_two_batches_on_a_fresh_context(dl):
    """The second launch finds the tensor memory the first one freed."""
    ctx = dl.Context(0)
    rng = np.random.RandomState(7200)
    n = _sm_count() * 2 + 3
    for seed in (8, 9):
        data, off, ln = _batch(seed, _lens(rng, n))
        _assert_like_oracle(dl, data, off, ln, ctx=ctx)
