"""Decoder parity on synthetic and corrupted LZ4 streams.

The compressors only ever emit greedy streams, so the decoder suite never saw long length runs, literal runs of more than
4 KiB inside a compressed block, tokens on the copy-form bounds of the block decoder, matches that start at dictionary
byte 0 or straddle the dictionary and the output, or blocks that end right after a match.  This file writes such streams
sequence by sequence (`BlockWriter`, pure Python, with a byte-by-byte model decoder), wraps them in frames, derives
corrupt inputs from them, and sends everything through every decode route of the library: the bytes, lengths and
statuses must equal the oracle's.

Two documented deviations of the library from the reference's decompressBuffer are modelled by `frame_model`, and each
is pinned by a test of its own:
  * an independent block's history is the dictionary only (the reference lets block k read block k - 1 when the frame
    declares its content size);
  * a block never decodes past blockMaxSize (the LZ4 frame format's limit, which liblz4 enforces too).

CPU tests (no marker) pin the generator against the oracle and liblz4; the GPU tests carry `@pytest.mark.gpu`.
"""
import ctypes as C
import os
import struct

import numpy as np
import pytest

import oracle

OK, TOO_SMALL, MALFORMED, OFFSET_ZERO, DICT_OOB = 0, 1, 2, 3, 4
BLOCK_MAX = {4: 65536, 5: 262144, 6: 1048576, 7: 4194304}


# ================================================================================ stream generator
def _ext(n):
    """Length bytes behind a nibble of 15 for a length n >= 15: 255 * k + r."""
    n -= 15
    out = bytearray()
    while n >= 255:
        out.append(255)
        n -= 255
    out.append(n)
    return bytes(out)


class BlockWriter(object):
    """Writes one LZ4 block sequence by sequence while a model decoder follows: literals are appended, a match is copied
    byte by byte (forward, any overlap) from history ++ output.  `history` is what precedes the block's output: the
    dictionary, plus the frame's earlier output for a linked block."""

    def __init__(self, history=b""):
        self.h = len(history)
        self.buf = bytearray(history)
        self.comp = bytearray()
        self.last_match_end = None          # block-relative output position where the last match ended
        self.final_lits = None              # length of the closing literal run (None: the block ends after a match)

    @property
    def pos(self):
        return len(self.buf) - self.h

    @property
    def out(self):
        return bytes(self.buf[self.h:])

    def token_bytes(self, lit, ml, offset):
        L, m = len(lit), ml - 4
        t = bytearray([(min(L, 15) << 4) | min(m, 15)])
        if L >= 15:
            t += _ext(L)
        t += lit + struct.pack("<H", offset)
        if m >= 15:
            t += _ext(m)
        return t

    def seq(self, lit, ml, offset):
        lit = bytes(lit)
        assert ml >= 4 and 1 <= offset <= 65535
        self.comp += self.token_bytes(lit, ml, offset)
        self.buf += lit
        src = len(self.buf) - offset
        assert src >= 0, "the match would read before the history"
        if offset >= ml:
            self.buf += self.buf[src:src + ml]
        else:                                                        # overlapping forward copy = the period repeated
            period = bytes(self.buf[src:src + offset])
            self.buf += (period * (ml // offset + 1))[:ml]
        self.last_match_end = self.pos
        return self

    def end(self, lit=b""):
        """Closing literal run (possibly empty: a lone token 0x00)."""
        lit = bytes(lit)
        L = len(lit)
        self.comp.append(min(L, 15) << 4)
        if L >= 15:
            self.comp += _ext(L)
        self.comp += lit
        self.buf += lit
        self.final_lits = L
        return self

    @property
    def spec_ok(self):
        """LZ4 block format end conditions: the last 5 bytes are literals and the last match starts >= 12 bytes before the
        end (liblz4 enforces both)."""
        if self.final_lits is None or self.final_lits < 5:
            return False
        return self.last_match_end is None or self.pos - (self.last_match_end - 4) >= 12

    def block(self):
        return bytes(self.comp), self.out


def _rb(rng, n):
    return rng.randint(0, 256, n).astype(np.uint8).tobytes()


# length values the decoders treat differently: nibble only, nibble 15 with 1, 2 (255 then 0), 3 and more length bytes
# (3 or more force the serial form of the speculative window), and k = 1..4 runs of 255 with a remainder
SPECIAL_LENGTHS = [0, 1, 14, 15, 16, 15 + 254, 15 + 255, 15 + 255 + 9, 15 + 2 * 255 + 3, 15 + 3 * 255 + 1, 15 + 4 * 255 + 200]


def _pick_offset(rng, w, L, ml, dict_len):
    """A valid offset for a match whose literals L are about to be written: the period path, the merged-pass bound
    min(L + ml, 32) and one below it, 65535, a source at output index 0, at dictionary byte 0, straddling the two."""
    avail = w.h + w.pos + L                                         # bytes before the match's first output byte
    out0 = avail - dict_len                                         # offset whose source is output index 0
    b = min(L + ml, 32)
    cands = [int(rng.randint(1, 32)), b, b - 1, 65535, out0, avail, int(rng.randint(1, 4000))]
    if dict_len:
        cands += [avail - int(rng.randint(0, dict_len)), out0 + max(1, min(ml - 1, dict_len))]   # inside / straddling
    cands = [c for c in cands if 1 <= c <= min(avail, 65535)]
    return int(cands[rng.randint(len(cands))]) if cands else None


def random_block(rng, size, history=b"", dict_len=0, large=False, end="lits"):
    """A valid block of about `size` decoded bytes.  end: "lits" (a closing literal run of 0..40 bytes), "spec" (>= 12
    closing literals: liblz4 decodes it too), "match" (the block ends right after a match)."""
    w = BlockWriter(history)
    lens = SPECIAL_LENGTHS + ([5000, 70000] if large else [])
    while w.pos < size:
        L = int(rng.choice(lens)) if rng.randint(3) == 0 else int(rng.randint(0, 12))
        ml = 4 + (int(rng.choice(lens)) if rng.randint(3) == 0 else int(rng.randint(0, 20)))
        if w.h + w.pos + L == 0:
            L = 1
        off = _pick_offset(rng, w, L, ml, dict_len)
        if off is None:
            L, off = L + 1, 1
        w.seq(_rb(rng, L), ml, off)
    if end == "lits":
        w.end(_rb(rng, int(rng.choice([0, 1, 4, 5, 15, 40]))))
    elif end == "spec":
        w.end(_rb(rng, int(rng.randint(12, 60))))
    return w


def lengths_block(rng, which, history=b""):
    """Every special length on the literal run (which="lit") or on the match (which="match"), each in its own sequence."""
    w = BlockWriter(history)
    w.seq(_rb(rng, 40), 4, 1)
    for v in SPECIAL_LENGTHS:
        if which == "lit":
            w.seq(_rb(rng, v), 4 + int(rng.randint(0, 20)), int(rng.randint(1, 40)))
        else:
            w.seq(_rb(rng, int(rng.randint(0, 3))), 4 + v, int(rng.choice([1, 3, 17, 31, 32, 33, 40])))
    return w.end(_rb(rng, 12))


def quick_bound_block(rng, below_prob):
    """Runs of sequences of at most 32 bytes whose offsets sit exactly on the quick-form bound of the block decoder's
    window (offset == rel_o + lit + ml: the match source ends where the window's output starts) or one below it.  The
    windows are simulated as the decoder forms them: a window starts at a token and takes every token that starts within
    32 bytes of it."""
    toks = [(int(rng.randint(0, 15)), int(rng.randint(4, 19))) for _ in range(int(rng.randint(60, 200)))]
    head = 40
    size = [3 + L for L, _ in toks]
    w = BlockWriter()
    w.seq(_rb(rng, head), 4, 1)                                      # 44 bytes of history, a window of its own
    t = 0
    while t < len(toks):
        ip0, op0, k, rel = 0, w.pos, t, 0
        offs = []
        while k < len(toks) and ip0 < 32:
            L, ml = toks[k]
            off = rel + L + ml - (1 if rng.rand() < below_prob else 0)
            offs.append(off)
            ip0 += size[k]
            rel += L + ml
            k += 1
        for j, off in enumerate(offs):
            L, ml = toks[t + j]
            w.seq(_rb(rng, L), ml, off)
        assert w.pos >= op0
        t = k
    return w.end(_rb(rng, 16))


def slow_window_block(rng):
    """The first token the speculative window cannot size (a length run of 3 or more bytes) at every position p of a
    window: the window starts behind the previous slow token, p bytes of short sequences, then the slow token.
    (Sequences are >= 3 bytes, so p = 1 and p = 2 cannot start a token.)"""
    w = BlockWriter()
    w.seq(_rb(rng, 64), 4, 1)
    long_run = 15 + 3 * 255 + 7
    for p in [0] + list(range(3, 32)):
        rest = p
        while rest:
            s = rest if rest <= 17 else min(17, rest - 3)
            w.seq(_rb(rng, s - 3), int(rng.randint(4, 19)), int(rng.randint(1, 60)))
            rest -= s
        if p % 2:
            w.seq(_rb(rng, long_run), 4, int(rng.randint(1, 60)))
        else:
            w.seq(_rb(rng, 1), 4 + long_run, int(rng.randint(1, 60)))
    return w.end(_rb(rng, 12))


def dict_block(rng, dictionary):
    """Matches entirely inside the dictionary (from its byte 0 on), straddling it and the output, at output index 0."""
    D = len(dictionary)
    w = BlockWriter(dictionary)
    w.seq(b"", min(D, 20), min(D, 65535))                            # dictionary byte 0 (the farthest byte in reach)
    w.seq(_rb(rng, 3), 4 + int(rng.randint(0, 30)), w.pos + 3 + 1 + int(rng.randint(0, min(D, 65000) - 1)))
    w.seq(_rb(rng, 2), min(D, 10) + 8, w.pos + 2 + min(D, 10))       # straddles the dictionary's end and the output
    w.seq(_rb(rng, 1), 6, w.pos + 1)                                 # source = output index 0
    for _ in range(20):
        L = int(rng.randint(0, 20))
        ml = 4 + int(rng.choice(SPECIAL_LENGTHS))
        w.seq(_rb(rng, L), ml, _pick_offset(rng, w, L, ml, D))
    return w.end(_rb(rng, 12))


def capacity_cases(w):
    """[(block, cap)] for a capacity of exactly the decoded size and of one byte less; the shortfall lies in the closing
    literals or, for a block that ends after a match, in the match."""
    comp, out = w.block()
    return [(comp, len(out)), (comp, len(out) - 1)] if len(out) else [(comp, 0)]


# ================================================================================ frames
def build_frame(blocks, bd, linked, content_size=None, dict_id=None, content=None, block_checksum=False):
    """blocks: [(payload, stored)].  content_size: the declared size or None; content: the bytes whose xxh32 closes the
    frame (None: no content checksum)."""
    flg = 0x40 | (0 if linked else 0x20) | (0x08 if content_size is not None else 0) | (0x04 if content is not None else 0)
    flg |= (0x10 if block_checksum else 0) | (0x01 if dict_id is not None else 0)
    desc = bytes([flg, bd << 4])
    if content_size is not None:
        desc += struct.pack("<Q", content_size)
    if dict_id is not None:
        desc += struct.pack("<I", dict_id)
    out = bytearray(struct.pack("<I", 0x184D2204) + desc + bytes([(oracle.xxh32(desc) >> 8) & 0xFF]))
    for payload, stored in blocks:
        out += struct.pack("<I", len(payload) | (0x80000000 if stored else 0)) + payload
        if block_checksum:
            out += struct.pack("<I", oracle.xxh32(payload))
    out += struct.pack("<I", 0)
    if content is not None:
        out += struct.pack("<I", oracle.xxh32(content))
    return bytes(out)


class Frame(object):
    """A frame together with what built it, so that corrupt variants can be rebuilt around mutated blocks."""

    def __init__(self, blocks, bd, linked, dictionary=b"", with_size=True, cc=False, plain=None, content_size=None):
        self.blocks, self.bd, self.linked, self.dictionary = list(blocks), bd, linked, dictionary
        self.with_size, self.cc, self.plain = with_size, cc, plain
        self.content_size = content_size if content_size is not None else (len(plain) if with_size else None)

    @property
    def B(self):
        return BLOCK_MAX[self.bd]

    def bytes(self):
        return build_frame(self.blocks, self.bd, self.linked, self.content_size,
                           oracle.xxh32(self.dictionary) if self.dictionary else None, self.plain if self.cc else None)

    def with_blocks(self, blocks):
        return Frame(blocks, self.bd, self.linked, self.dictionary, self.with_size, False, self.plain, self.content_size)


def parse_frame(f, dictionary=b""):
    """The Frame of well-formed frame bytes (no block checksums), for frame_model(..., verify_checksum=False)."""
    flg, bd = f[4], (f[5] >> 4) & 7
    pos, size = 6, None
    if flg & 0x08:
        size = struct.unpack_from("<Q", f, pos)[0]
        pos += 8
    pos += 4 * (flg & 1) + 1
    blocks = []
    while True:
        bs = struct.unpack_from("<I", f, pos)[0]
        pos += 4
        if bs == 0:
            break
        blocks.append((bytes(f[pos:pos + (bs & 0x7FFFFFFF)]), bool(bs >> 31)))
        pos += bs & 0x7FFFFFFF
    return Frame(blocks, bd, not flg & 0x20, dictionary, size is not None, False, None, content_size=size)


def random_frame(rng, bd, linked, nblocks, dictionary=b"", with_size=True, cc=False, stored_every=0, large=False,
                 full=True, lit_heavy=False):
    """nblocks valid blocks of at most blockMaxSize each (full=True: inner blocks exactly blockMaxSize).  A linked block's
    matches reach into the earlier blocks and the dictionary; an independent block's into the dictionary only."""
    B = BLOCK_MAX[bd]
    out = bytearray()
    blocks = []
    lens = SPECIAL_LENGTHS + ([5000, 70000] if large else [])
    for k in range(nblocks):
        want = B if full and k + 1 < nblocks else int(rng.randint(1, B + 1))
        if stored_every and k % stored_every == stored_every - 1:
            raw = _rb(rng, want)
            blocks.append((raw, True))
            out += raw
            continue
        hist = dictionary + bytes(out[-65536:]) if linked else dictionary
        # offsets only reach 65535 back: a longer history is cut, and then output index 0 is out of reach anyway
        dl = len(dictionary) if (not linked or len(out) <= 65536) else 0
        if linked and len(out) > 65536:
            hist = hist[-65536:]
        w = BlockWriter(hist)
        while True:
            if lit_heavy:
                L, ml = int(rng.choice([300, 5000, 70000])), 4 + int(rng.choice([0, 16, 300]))
            else:
                L = int(rng.choice(lens)) if rng.randint(3) == 0 else int(rng.randint(0, 12))
                ml = 4 + (int(rng.choice(lens)) if rng.randint(3) == 0 else int(rng.randint(0, 20)))
            if w.pos + L + ml + 40 > want:
                break
            if w.h + w.pos + L == 0:
                L = 1
            off = _pick_offset(rng, w, L, ml, dl)
            if off is None:
                L, off = L + 1, 1
            w.seq(_rb(rng, L), ml, off)
        w.end(_rb(rng, want - w.pos))
        comp, dec = w.block()
        blocks.append((comp, False))
        out += dec
    return Frame(blocks, bd, linked, dictionary, with_size, cc, bytes(out))


def frame_model(fr, verify_checksum=True):
    """What every frame route of the library returns: the decoded bytes, or the status of the first error (an int).
    The oracle's block decoder per block, sequentially like bufferDecompress.js:133-192, with the library's two
    deviations: an independent block's history is the dictionary only, and a block never decodes past blockMaxSize."""
    B = fr.B
    if fr.content_size:
        cap_total = fr.content_size
    else:
        cap_total = sum(len(p) if s else min(len(p) * 255, B) for p, s in fr.blocks)
    out = np.zeros(cap_total + 1, dtype=np.uint8)
    d = fr.dictionary or None
    pos = 0
    for payload, stored in fr.blocks:
        room = min(B, cap_total - pos)
        if stored:
            if len(payload) > room:
                return TOO_SMALL
            out[pos:pos + len(payload)] = np.frombuffer(payload, dtype=np.uint8)
            n = len(payload)
        else:
            try:
                if fr.linked:
                    n = oracle.decompress_block(payload, 0, len(payload), out[:pos + room], pos, d)
                else:
                    tmp = np.zeros(room, dtype=np.uint8)
                    n = oracle.decompress_block(payload, 0, len(payload), tmp, 0, d)
                    out[pos:pos + n] = tmp[:n]
            except oracle.OracleError as e:
                return -e.code
        pos += n
    got = out[:pos].tobytes()
    if fr.cc and verify_checksum and oracle.xxh32(got) != oracle.xxh32(fr.plain):
        return 7
    return got


# ================================================================================ mutator
def mutations(rng, comp, exhaustive):
    """Corrupt variants of one compressed block: prefixes (truncation), byte flips, zeroed stretches, an offset set to 0 or
    past the history, a length run extended to the end of the input.  exhaustive: every prefix and a flip at every
    position; otherwise a random sample of each."""
    comp = bytes(comp)
    n = len(comp)
    cut = range(n) if exhaustive else sorted(set(int(x) for x in rng.randint(0, max(n, 1), 24)))
    out = [comp[:k] for k in cut]
    for k in (range(n) if exhaustive else rng.randint(0, max(n, 1), 48)):
        b = bytearray(comp)
        if n:
            b[k] ^= int(rng.randint(1, 256))
            out.append(bytes(b))
    for _ in range(8):
        if n:
            a = int(rng.randint(0, n))
            e = min(n, a + int(rng.randint(1, 64)))
            b = bytearray(comp)
            b[a:e] = bytes(e - a)
            out.append(bytes(b))
    # token-aware edits: walk the tokens and edit the offset / length bytes of a few
    toks = _token_positions(comp)
    for t in (toks if exhaustive else [toks[i] for i in rng.randint(0, len(toks), min(len(toks), 6))]) if toks else []:
        tok, offpos, mlpos = t
        if offpos is not None:
            b = bytearray(comp)
            b[offpos:offpos + 2] = b"\x00\x00"
            out.append(bytes(b))
            b = bytearray(comp)
            b[offpos:offpos + 2] = b"\xff\xff"
            out.append(bytes(b))
        b = bytearray(comp)                                          # literal run of 15 whose length bytes never end
        b[tok] |= 0xF0
        out.append(bytes(b[:tok + 1]) + b"\xff" * (n - tok - 1))
        if offpos is not None:
            b = bytearray(comp)                                      # match length run that never ends
            b[tok] |= 0x0F
            out.append(bytes(b[:offpos + 2]) + b"\xff" * (n - offpos - 2))
    return out


def _token_positions(comp):
    """[(token position, offset position or None, match length position)] of a well-formed block."""
    res, ip, n = [], 0, len(comp)
    while ip < n:
        tok = ip
        t = comp[ip]
        ip += 1
        L = t >> 4
        if L == 15:
            while ip < n:
                v = comp[ip]
                ip += 1
                L += v
                if v != 255:
                    break
        ip += L
        if ip >= n:
            res.append((tok, None, None))
            break
        offpos = ip
        ip += 2
        if (t & 15) == 15:
            while ip < n:
                v = comp[ip]
                ip += 1
                if v != 255:
                    break
        res.append((tok, offpos, ip))
    return res


# ================================================================================ targeted error builders
def _history_frame(rng, nblocks, bd=5):
    """A linked frame of literal-heavy blocks (>= 256 KiB so that the jump decoder takes it)."""
    return random_frame(rng, bd, True, nblocks, with_size=True)


def case_a(rng):
    """Token t1 reads before the history; a later token t2 of the same block is malformed (the reference: DICT_OOB)."""
    fr = _history_frame(rng, 3)
    w = BlockWriter()
    w.comp += w.token_bytes(_rb(rng, 5), 8, 65535)                   # block 0: 5 bytes of output, offset 65535
    w.comp += bytes([0xF0]) + b"\xff" * 3                            # t2: a literal run whose length bytes end the input
    blocks = [(bytes(w.comp), False)] + fr.blocks[1:]
    return Frame(blocks, fr.bd, True, b"", True, False, fr.plain)


def case_a_later_block(rng):
    """The same in block 1 of a linked frame behind a short block 0: t1 reads before output index 0, t2 has offset 0."""
    fr = _history_frame(rng, 3)
    b0 = random_block(rng, 1000)
    n0 = b0.pos
    t1 = BlockWriter().token_bytes(_rb(rng, 3), 4, n0 + 3 + 50)
    t2 = bytearray(BlockWriter().token_bytes(_rb(rng, 2), 4, 1))
    t2[-2:] = b"\x00\x00"                                           # offset 0
    blk1 = bytes(t1) + bytes(t2) + bytes([0x10]) + b"z"
    blocks = [(b0.block()[0], False), (blk1, False)] + fr.blocks[1:]
    return Frame(blocks, fr.bd, True, b"", True, False, b0.out + fr.plain)


def case_b(rng):
    """One token both reads before the history and overflows the block (the reference: DICT_OOB)."""
    fr = _history_frame(rng, 3)
    w = BlockWriter()
    w.comp += w.token_bytes(_rb(rng, 5), 4 + fr.B, 65535)            # a match of blockMaxSize + 4 bytes
    w.comp += bytes([0x10]) + b"z"
    blocks = [(bytes(w.comp), False)] + fr.blocks[1:]
    return Frame(blocks, fr.bd, True, b"", True, False, fr.plain)


def case_c(rng):
    """The declared content size is too small, an early token exceeds it, a later token reads before the history
    (the reference: OUTPUT_TOO_SMALL)."""
    fr = _history_frame(rng, 3)
    w = BlockWriter()
    w.seq(_rb(rng, 2000), 4, 1)                                      # past the declared 1000 bytes
    w.comp += w.token_bytes(b"ab", 4, 65535)                         # reads before output index 0
    w.comp += bytes([0x10]) + b"z"
    blocks = [(bytes(w.comp), False)] + fr.blocks[1:]
    return Frame(blocks, fr.bd, True, b"", True, False, fr.plain, content_size=1000)


# ================================================================================ CPU: the generator itself
def _blocks_for_batch(rng, dictionary=b""):
    """(writer, dictionary-or-None) for every kind of synthetic block."""
    ws = [lengths_block(rng, "lit"), lengths_block(rng, "match"), slow_window_block(rng), quick_bound_block(rng, 0.0),
          quick_bound_block(rng, 0.3), quick_bound_block(rng, 1.0), BlockWriter().end(b""), BlockWriter().end(_rb(rng, 7))]
    for end in ("lits", "spec", "match"):
        for size in (1, 40, 3000, 30000):
            ws.append(random_block(rng, size, end=end))
    if dictionary:
        ws += [dict_block(rng, dictionary) for _ in range(6)]
        ws += [random_block(rng, 2000, dictionary, len(dictionary), end=e) for e in ("lits", "match")]
    return ws


def test_generator_blocks_decode_as_modelled():
    import lz4f
    rng = np.random.RandomState(1)
    for dictionary in (b"", _rb(rng, 70000), _rb(rng, 300)):
        for w in _blocks_for_batch(rng, dictionary):
            comp, out = w.block()
            buf = np.zeros(len(out), dtype=np.uint8)
            assert oracle.decompress_block(comp, 0, len(comp), buf, 0, dictionary or None) == len(out)
            assert buf.tobytes() == out
            if w.spec_ok and lz4f.available():
                assert lz4f.decompress_block(comp, len(out), dictionary or None) == out
            if len(out):                                             # one byte less: the reference's capacity error
                with pytest.raises(oracle.OracleError) as ei:
                    oracle.decompress_block(comp, 0, len(comp), np.zeros(len(out) - 1, dtype=np.uint8), 0, dictionary or None)
                assert ei.value.code == oracle.E_OUTPUT_TOO_SMALL


def test_generator_reaches_the_special_shapes():
    rng = np.random.RandomState(2)
    comp, _ = slow_window_block(rng).block()
    runs = [len(comp[t:]) for t, _, _ in _token_positions(comp)]
    assert len(runs) > 40
    # every special length appears as a literal run and as a match length
    for which in ("lit", "match"):
        comp, _ = lengths_block(rng, which).block()
        assert b"\xff\xff\xff\xff" in comp and b"\xff\x00" in comp
    lb = random_block(rng, 300000, large=True)
    assert lb.pos > 65536


@pytest.mark.parametrize("linked", [False, True])
def test_generator_frames_match_the_reference(linked):
    rng = np.random.RandomState(3 + linked)
    for bd, nb, kw in [(4, 5, {}), (5, 3, dict(stored_every=2)), (6, 2, dict(with_size=False, cc=True, large=True)),
                       (7, 1, dict(full=False)), (4, 4, dict(dictionary=_rb(rng, 5000), cc=True)),
                       (5, 2, dict(dictionary=_rb(rng, 80000), with_size=False))]:
        fr = random_frame(rng, bd, linked, nb, **kw)
        f = fr.bytes()
        assert frame_model(fr) == fr.plain, (bd, nb, kw)
        if linked or not kw.get("dictionary") or nb == 1:
            # an independent block behind the first one reads the dictionary; the reference gives it the earlier output
            assert oracle.decompress_buffer(f, kw.get("dictionary")) == fr.plain, (bd, nb, kw)


def test_targeted_error_frames_name_the_reference_errors():
    rng = np.random.RandomState(4)
    for build, want in ((case_a, DICT_OOB), (case_a_later_block, DICT_OOB), (case_b, DICT_OOB), (case_c, TOO_SMALL)):
        fr = build(rng)
        with pytest.raises(oracle.OracleError) as ei:
            oracle.decompress_buffer(fr.bytes())
        assert -ei.value.code == want, build.__name__
        assert frame_model(fr) == want, build.__name__


def test_mutator_reaches_every_block_error():
    rng = np.random.RandomState(5)
    seen = set()
    for w in (lengths_block(rng, "lit"), random_block(rng, 200), quick_bound_block(rng, 0.5)):
        comp, out = w.block()
        for m in mutations(rng, comp, exhaustive=len(comp) < 400):
            try:
                oracle.decompress_block(m, 0, len(m), np.zeros(len(out) + 64, dtype=np.uint8), 0)
                seen.add(OK)
            except oracle.OracleError as e:
                seen.add(-e.code)
    assert seen == {OK, TOO_SMALL, MALFORMED, OFFSET_ZERO, DICT_OOB}


# ================================================================================ GPU: every decode route
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
def frame_ctxs(dl):
    """The frame decoders, each forced: k_decompress_chain, the jump decoder with its chunked scan (blocks > 64 KiB) or the
    warp scan, and the serial scan everywhere."""
    return {"default": dl.default_context(),
            "chain": _ctx(dl, DLZ4_JUMP_MIN_KIB=str(1 << 30)),
            "jump": _ctx(dl, DLZ4_JUMP_MIN_KIB="0"),
            "serial": _ctx(dl, DLZ4_JUMP_MIN_KIB="0", DLZ4_JD_SERIAL_SCAN="1")}


def _want(model):
    return model if isinstance(model, bytes) else (model, oracle.MESSAGES[-model])


def _frame_result(dl, ctx, f, dictionary):
    try:
        return dl.decompressBuffer(f, dictionary or None, True, False, ctx=ctx)
    except dl.LZ4Error as e:
        return (e.status, str(e))


def _check_frame(dl, ctxs, fr, tag):
    f = fr.bytes()
    want = _want(frame_model(fr))
    for name, ctx in ctxs.items():
        got = _frame_result(dl, ctx, f, fr.dictionary)
        assert got == want, (tag, name, got if isinstance(got, tuple) else len(got),
                             want if isinstance(want, tuple) else len(want))


def _pack(cases):
    """[(comp, cap)] -> src, off, len, dst_off, cap (16 bytes between output slots)."""
    lens = np.array([len(c) for c, _ in cases], dtype=np.uint32)
    caps = np.array([cap for _, cap in cases], dtype=np.uint32)
    off = np.zeros(len(cases), dtype=np.uint64)
    off[1:] = np.cumsum(lens.astype(np.uint64))[:-1]
    doff = np.zeros(len(cases), dtype=np.uint64)
    doff[1:] = np.cumsum(caps.astype(np.uint64) + 16)[:-1]
    src = np.frombuffer(b"".join(c for c, _ in cases) + bytes(16), dtype=np.uint8)
    return src, off, lens, doff, caps


def _check_batch(got, want, tag):
    _, glen, gst = got
    _, olen, ost = want
    assert np.array_equal(gst.astype(np.int32), -ost), (tag, np.nonzero(gst.astype(np.int32) != -ost)[0][:10])
    ok = ost == 0
    assert np.array_equal(glen[ok], olen[ok]), tag


def _check_bytes(got, want, doff, tag):
    gdst, glen, gst = got
    odst, olen, ost = want
    for i in np.nonzero(ost == 0)[0]:
        a, n = int(doff[i]), int(olen[i])
        assert gdst[a:a + n].tobytes() == odst[a:a + n].tobytes(), (tag, int(i))


def _dev_call(dl, ctx, src, off, lens, doff, caps, dictionary=None, hist=0, dst_init=None):
    """dlz4_decompress_blocks_dev on torch tensors; returns (dst, out_len, status) as numpy without raising."""
    import torch
    from divortio_lz4_b200 import api
    dev = torch.device("cuda", 0)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).astype(dt)).to(dev)
    total = int((doff + caps).max())
    dst = t(dst_init if dst_init is not None else np.zeros(total + 16, dtype=np.uint8), np.uint8)
    n = len(lens)
    ol = torch.zeros(n, dtype=torch.int32, device=dev)
    st = torch.zeros(n, dtype=torch.uint8, device=dev)
    ts, to, tl, tdo, tc = t(src, np.uint8), t(off, np.int64), t(lens, np.int32), t(doff, np.int64), t(caps, np.int32)
    td = t(np.frombuffer(dictionary, dtype=np.uint8), np.uint8) if dictionary else None
    p = lambda x: C.c_void_p(x.data_ptr()) if x is not None and x.numel() else None
    r = api.lib().dlz4_decompress_blocks_dev(ctx.handle, p(ts), p(to), p(tl), n, p(dst), p(tdo), p(tc), p(td),
                                             len(dictionary) if dictionary else 0, hist, p(ol), p(st), C.c_void_p(1))
    torch.cuda.synchronize()
    assert r < 20, r
    return dst.cpu().numpy(), ol.cpu().numpy().astype(np.uint32), st.cpu().numpy()


def _batch_routes(dl, src, off, lens, doff, caps, dictionary, packed_ctx):
    d = dictionary or None
    yield "strided", dl.decompress_blocks(src, off, lens, doff, caps, d, check=False)
    if len(src) - 16 == int(lens.sum()):
        yield "packed", dl.decompress_blocks(src[:int(lens.sum())], None, lens, doff, caps, d, ctx=packed_ctx, check=False)
    yield "dev", _dev_call(dl, dl.default_context(), src, off, lens, doff, caps, dictionary)


@pytest.fixture(scope="module")
def packed_ctx(dl):
    return _ctx(dl, DLZ4_CHUNK_MIB="1")                              # 1 MiB chunks: every batch here spans several


@pytest.mark.gpu
@pytest.mark.parametrize("with_dict", [False, True])
def test_synthetic_blocks_every_batch_route(dl, packed_ctx, with_dict):
    """k_decompress_blocks<false / true> on the strided, packed (several chunks) and device-resident routes; each block at
    capacity exactly its decoded size and one byte less; the batch repeated to >= 1024 blocks."""
    rng = np.random.RandomState(10 + with_dict)
    dictionary = _rb(rng, 70000) if with_dict else b""
    cases = []
    for w in _blocks_for_batch(rng, dictionary):
        cases += capacity_cases(w)
    for reps in (1, 1024 // len(cases) + 1):
        src, off, lens, doff, caps = _pack(cases * reps)
        want = oracle.decompress_blocks(src, off, lens, doff, caps, dictionary or None)
        assert (want[2] == 0).sum() and (want[2] == oracle.E_OUTPUT_TOO_SMALL).sum()
        for name, got in _batch_routes(dl, src, off, lens, doff, caps, dictionary, packed_ctx):
            _check_batch(got, want, (name, reps))
            _check_bytes(got, want, doff, (name, reps))


@pytest.mark.gpu
def test_corrupt_blocks_report_the_reference_status(dl, packed_ctx):
    """Every prefix and a flip at every byte of short blocks, random edits of longer ones, zeroed stretches, offsets of 0
    and past the history, length runs to the end of the input: per-block status == the oracle's."""
    rng = np.random.RandomState(20)
    dictionary = _rb(rng, 3000)
    for d in (b"", dictionary):
        cases = []
        for w in [lengths_block(rng, "lit"), random_block(rng, 300), random_block(rng, 300, end="match"),
                  quick_bound_block(rng, 0.5), slow_window_block(rng), random_block(rng, 20000)] + \
                 ([dict_block(rng, d)] if d else []):
            comp, out = w.block()
            for m in mutations(rng, comp, exhaustive=len(comp) < 600):
                cases.append((m, len(out) + 64))
        src, off, lens, doff, caps = _pack(cases)
        want = oracle.decompress_blocks(src, off, lens, doff, caps, d or None)
        for code in (0, oracle.E_MALFORMED, oracle.E_OFFSET_ZERO, oracle.E_DICT_OOB):
            assert (want[2] == code).any(), code
        for name, got in _batch_routes(dl, src, off, lens, doff, caps, d, packed_ctx):
            _check_batch(got, want, (name, len(d)))
            _check_bytes(got, want, doff, (name, len(d)))


def _large_blocks(rng, B, n):
    ws = []
    for k in range(n):
        w = random_block(rng, B - 80000, large=True, end="lits" if k % 2 else "match")
        if w.pos > B:
            w = random_block(rng, B // 2, large=True)
        ws.append(w)
    return ws


@pytest.mark.gpu
def test_large_uniform_blocks_take_the_jump_route_and_its_fallback(dl):
    """Uniform power-of-two blocks > 64 KiB, fewer than 1024, no dictionary: the batch call's jump decoder (host and
    device-resident); one corrupt block sends the batch to one warp per block, which must name each block's status."""
    rng = np.random.RandomState(30)
    B = 262144
    ws = _large_blocks(rng, B, 6)
    assert max(w.pos for w in ws) > 65536
    cases = [(w.block()[0], B) for w in ws]
    for corrupt in (False, True):
        cs = list(cases)
        if corrupt:
            comp = bytearray(cs[3][0])
            toks = [t for t in _token_positions(bytes(comp)) if t[1] is not None]
            offpos = toks[len(toks) // 2][1]
            comp[offpos:offpos + 2] = b"\x00\x00"                     # offset 0 in the middle of block 3
            cs[3] = (bytes(comp), B)
        src, off, lens, _, caps = _pack(cs)
        doff = np.arange(len(cs), dtype=np.uint64) * B
        want = oracle.decompress_blocks(src, off, lens, doff, caps)
        assert (want[2] != 0).any() == corrupt
        for name, got in (("host", dl.decompress_blocks(src, off, lens, doff, caps, check=False)),
                          ("dev", _dev_call(dl, dl.default_context(), src, off, lens, doff, caps))):
            _check_batch(got, want, (name, corrupt))
            _check_bytes(got, want, doff, (name, corrupt))


# ---------------------------------------------------------------- frames
def _frames(rng):
    yield "linked64k", random_frame(rng, 4, True, 6, stored_every=4)
    yield "linked64k_short", random_frame(rng, 4, True, 3, full=False)
    yield "linked256k_dict", random_frame(rng, 5, True, 3, dictionary=_rb(rng, 70000), cc=True)
    yield "linked1m_nosize", random_frame(rng, 6, True, 2, with_size=False, large=True)
    yield "linked4m", random_frame(rng, 7, True, 1, full=False, large=True)
    yield "indep64k", random_frame(rng, 4, False, 8, stored_every=3, cc=True, with_size=False)
    yield "indep256k_dict", random_frame(rng, 5, False, 3, dictionary=_rb(rng, 1000))
    yield "indep1m_short", random_frame(rng, 6, False, 3, full=False, large=True)


@pytest.mark.gpu
def test_synthetic_frames_on_every_frame_decoder(dl, frame_ctxs):
    rng = np.random.RandomState(40)
    for tag, fr in _frames(rng):
        _check_frame(dl, frame_ctxs, fr, tag)


@pytest.mark.gpu
@pytest.mark.parametrize("linked", [True, False])
def test_frame_of_8_mib_and_more_overlaps_its_group_copies(dl, frame_ctxs, linked):
    """>= 8 MiB of frame: the chunked scan starts on groups of blocks as they land."""
    rng = np.random.RandomState(41 + linked)
    fr = random_frame(rng, 5, linked, 36, lit_heavy=True, cc=True)
    assert len(fr.bytes()) >= 8 << 20
    _check_frame(dl, {k: frame_ctxs[k] for k in ("default", "serial")}, fr, "8mib")


@pytest.mark.gpu
def test_corrupt_frames_agree_on_every_decoder(dl, frame_ctxs):
    """Corrupt blocks inside otherwise valid frames: the same bytes or the same error (status and message) on the chain
    kernel, the serial scan and the chunked scan, and that result is the reference's."""
    rng = np.random.RandomState(50)
    for tag, fr in _frames(rng):
        for k, (payload, stored) in enumerate(fr.blocks):
            if stored:
                continue
            for m in mutations(rng, payload, exhaustive=False)[::7]:
                blocks = list(fr.blocks)
                blocks[k] = (m, False)
                _check_frame(dl, frame_ctxs, fr.with_blocks(blocks), (tag, k))


@pytest.mark.gpu
@pytest.mark.parametrize("case", [case_a, case_a_later_block, case_b, case_c])
def test_history_errors_keep_the_reference_order(dl, frame_ctxs, case):
    """(a) a token reads before the history and a later one is malformed, (b) one token reads before the history and
    overflows the block, (c) the declared size is exceeded before a token reads before the history: the jump decoder
    must name the error the reference names first."""
    rng = np.random.RandomState(60)
    fr = case(rng)
    assert len(fr.bytes()) >= 256 << 10
    with pytest.raises(oracle.OracleError) as ei:
        oracle.decompress_buffer(fr.bytes())
    assert frame_model(fr) == -ei.value.code
    _check_frame(dl, frame_ctxs, fr, case.__name__)


@pytest.mark.gpu
def test_independent_block_history_is_the_dictionary_only(dl, frame_ctxs):
    """Deviation: block 1 of an independent frame reads block 0's output.  The reference decodes it (its output array is
    the whole frame's); the library gives an independent block the dictionary only (LZ4 frame format)."""
    rng = np.random.RandomState(70)
    for bd, B in ((4, 65536), (5, 262144)):
        b0 = BlockWriter().seq(_rb(rng, 100), 4, 1).end(_rb(rng, B - 104))
        w = BlockWriter(b0.out)
        w.seq(_rb(rng, 10), 8, 40).end(_rb(rng, 12))                 # reads 30 bytes before its own start
        fr = Frame([(b0.block()[0], False), (w.block()[0], False)], bd, False, b"", True, False, b0.out + w.out)
        assert oracle.decompress_buffer(fr.bytes()) == fr.plain
        assert frame_model(fr) == DICT_OOB
        _check_frame(dl, frame_ctxs, fr, bd)


@pytest.mark.gpu
def test_block_never_decodes_past_block_max_size(dl, frame_ctxs):
    """Deviation: a block that decodes to blockMaxSize + 1 bytes is "Output Buffer Too Small" on every decoder (the
    reference sizes its output by the declared content size only)."""
    rng = np.random.RandomState(80)
    for bd, linked, nblocks in ((4, True, 2), (4, True, 6), (5, True, 2), (4, False, 3), (5, False, 2)):
        fr = random_frame(rng, bd, linked, nblocks)
        w = BlockWriter(fr.plain[-65536:] if linked else b"")
        w.seq(_rb(rng, 8), fr.B - 8 + 1 - 5, 1).end(_rb(rng, 5))
        blocks = fr.blocks[:-1] + [(w.block()[0], False)]
        big = Frame(blocks, bd, linked, b"", True, False, fr.plain + bytes(w.out))
        assert len(oracle.decompress_buffer(big.bytes())) == len(big.plain)
        assert frame_model(big) == TOO_SMALL
        _check_frame(dl, frame_ctxs, big, (bd, linked, nblocks))


# ---------------------------------------------------------------- frame history in the batch call
def _hist_frame_batch(rng, dictionary, prefix_len):
    """Blocks that each read the gap in front of their slot, the caller's bytes before dst_off[0] and the dictionary:
    history = dictionary ++ dst[0..dst_off[i])."""
    blocks, doff, caps = [], [], []
    pos = prefix_len
    dst = bytearray(_rb(rng, prefix_len))
    for k in range(6):
        gap = 24 + 8 * k
        dst += _rb(rng, gap)
        pos += gap
        w = BlockWriter(dictionary + bytes(dst))
        w.seq(b"", 8, gap)                                           # the caller's bytes in the gap
        if prefix_len and pos < 60000:
            w.seq(b"", 5, w.h + w.pos - len(dictionary) - 1)         # dst[1]: before dst_off[0]
        if dictionary and pos < 60000:
            w.seq(_rb(rng, 1), 4, w.h + w.pos + 1)                   # dictionary byte 0
        w.seq(_rb(rng, 30), 40, 7).end(_rb(rng, 12))
        comp, out = w.block()
        blocks.append(comp)
        doff.append(pos)
        caps.append(len(out) + 5)
        dst += out + bytes(5)
        pos += len(out) + 5
    lens = np.array([len(b) for b in blocks], dtype=np.uint32)
    off = np.zeros(len(blocks), dtype=np.uint64)
    off[1:] = np.cumsum(lens.astype(np.uint64))[:-1]
    src = np.frombuffer(b"".join(blocks), dtype=np.uint8)
    return src, off, lens, np.array(doff, dtype=np.uint64), np.array(caps, dtype=np.uint32), bytes(dst[:prefix_len])


def _hist_model(src, off, lens, doff, caps, dictionary, init):
    dst = np.zeros(int((doff + caps).max()), dtype=np.uint8)
    dst[:len(init)] = np.frombuffer(init, dtype=np.uint8)
    out_len = np.zeros(len(lens), dtype=np.uint32)
    for i in range(len(lens)):
        out_len[i] = oracle.decompress_block(src, int(off[i]), int(lens[i]), dst[:int(doff[i] + caps[i])], int(doff[i]),
                                             dictionary or None)
    return dst, out_len


def _dirty(dl, ctx, nbytes):
    """An unrelated decode that leaves non-zero bytes all over the context's output scratch."""
    rng = np.random.RandomState(99)
    w = BlockWriter().end(_rb(rng, nbytes))
    comp, out = w.block()
    got = dl.decompress_blocks(np.frombuffer(comp, dtype=np.uint8), [0], [len(comp)], [0], [len(out)], ctx=ctx)
    assert got[0].tobytes() == out


@pytest.mark.gpu
@pytest.mark.parametrize("with_dict", [False, True])
def test_hist_frame_history_is_the_callers_dst(dl, with_dict):
    """DLZ4_HIST_FRAME: every byte of dst before a block is history, the caller's own bytes included, on the host strided,
    host packed and device-resident routes -- also on a context whose scratch an earlier decode has dirtied."""
    rng = np.random.RandomState(90 + with_dict)
    dictionary = _rb(rng, 2000) if with_dict else b""
    src, off, lens, doff, caps, _ = _hist_frame_batch(rng, dictionary, 0)
    want_dst, want_len = _hist_model(src, off, lens, doff, caps, dictionary, b"")
    ctx = _ctx(dl)
    _dirty(dl, ctx, int((doff + caps).max()) + 4096)
    for name, off_ in (("strided", off), ("packed", None)):
        dst, ol, st = dl.decompress_blocks(src, off_, lens, doff, caps, dictionary or None, dl.HIST_FRAME, ctx=ctx, check=False)
        assert not st.any() and np.array_equal(ol, want_len), name
        assert dst.tobytes() == want_dst.tobytes(), name
        _dirty(dl, ctx, int((doff + caps).max()) + 4096)
    dst, ol, st = _dev_call(dl, ctx, src, off, lens, doff, caps, dictionary, dl.HIST_FRAME)
    assert not st.any() and np.array_equal(ol, want_len)
    assert dst[:len(want_dst)].tobytes() == want_dst.tobytes()


@pytest.mark.gpu
def test_hist_frame_reads_the_callers_bytes_before_the_first_block(dl):
    """Through the C ABI with a caller-filled dst: history before dst_off[0] is the caller's, on a dirtied context too."""
    from divortio_lz4_b200 import api
    rng = np.random.RandomState(95)
    dictionary = _rb(rng, 500)
    src, off, lens, doff, caps, init = _hist_frame_batch(rng, dictionary, 5000)
    want_dst, want_len = _hist_model(src, off, lens, doff, caps, dictionary, init)
    ctx = _ctx(dl)
    for dirty in (False, True):
        if dirty:
            _dirty(dl, ctx, len(want_dst) + 4096)
        dst = np.zeros(len(want_dst), dtype=np.uint8)
        dst[:len(init)] = np.frombuffer(init, dtype=np.uint8)
        ol = np.zeros(len(lens), dtype=np.uint32)
        st = np.zeros(len(lens), dtype=np.uint8)
        d = np.frombuffer(dictionary, dtype=np.uint8)
        r = api.lib().dlz4_decompress_blocks(ctx.handle, src.ctypes.data, src.size, off.ctypes.data, lens.ctypes.data,
                                             len(lens), dst.ctypes.data, dst.size, doff.ctypes.data, caps.ctypes.data,
                                             d.ctypes.data, d.size, api.HIST_FRAME, ol.ctypes.data, st.ctypes.data)
        assert r == 0 and not st.any() and np.array_equal(ol, want_len), dirty
        assert dst.tobytes() == want_dst.tobytes(), dirty
