"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/dlz4_b200.h declares,
and the host-only logic (bounds, sharding, status text, frame header parsing) behaves.  No compute calls (no GPU here)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import divortio_lz4_b200 as dl
from divortio_lz4_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "dlz4_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dlz4_[a-z0-9_]+)\s*\(", text)))


def test_library_is_built_in_tree():
    assert os.path.exists(api.LIB_PATH), "run __graft_entry__.build()"
    assert os.path.dirname(api.LIB_PATH).startswith(ROOT)


def test_every_declared_symbol_is_exported():
    lib = C.CDLL(api.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), name
    assert set(declared) == set(api.EXPORTED_SYMBOLS)


def test_library_is_sm100a_only():
    import shutil
    import subprocess
    # the CUDA toolkit's bin directory need not be on PATH (the library's Makefile names nvcc by its full path too)
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", api.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_status_text_is_the_reference_text():
    L = api.lib()
    want = {1: "LZ4: Output Buffer Too Small", 2: "LZ4: Malformed Input", 3: "LZ4: Invalid Offset 0",
            4: "LZ4: Dictionary Offset Out of Bounds", 5: "LZ4: Invalid Magic Number", 6: "LZ4: Unsupported Version",
            7: "LZ4: Content Checksum Error"}
    for code, text in want.items():
        assert L.dlz4_strerror(code).decode() == text


def test_bounds():
    assert dl.compress_bound(0) == 16 and dl.compress_bound(65536) == 65536 + 257 + 16
    assert dl.frame_bound(0) >= 19 + 4 + 4


@pytest.mark.parametrize("n,world", [(0, 1), (1, 8), (7, 8), (8, 8), (10, 4), (16384, 8), (2048, 3), (1000003, 8)])
def test_shard_range_is_a_contiguous_partition(n, world):
    nxt = 0
    for r in range(world):
        first, count = dl.shard_range(n, world, r)
        assert first == nxt
        nxt = first + count
        for i in (first, first + count - 1):
            if count:
                assert (i * world) // n == r          # block i -> GPU floor(i*G/n)   (SURVEY 8e)
    assert nxt == n


def test_frame_info_parses_reference_golden_headers(kats):
    for k in kats["reference_golden"]["decode_frames"]:
        info = dl.frame_info(bytes.fromhex(k["hex"]))
        assert info.version == 1 and info.block_independence == 1
        assert info.nblocks == (1 if k["text"] else 0)
    with pytest.raises(dl.LZ4Error, match="Invalid Magic"):
        dl.frame_info(b"\x00" * 12)
    with pytest.raises(dl.LZ4Error, match="Unsupported Version 2"):
        dl.frame_info(bytes.fromhex("04224D18A0400000"))


def test_ensure_buffer_coercions():
    assert dl.ensureBuffer("hé").tobytes() == "hé".encode()
    assert dl.ensureBuffer([1, 2, 255]).tolist() == [1, 2, 255]
    assert dl.ensureBuffer({"a": 1}).tobytes() == b'{"a":1}'
    assert dl.ensureBuffer(np.arange(4, dtype=np.uint8)).tolist() == [0, 1, 2, 3]
    with pytest.raises(TypeError):
        dl.ensureBuffer(3.5)


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dl.Context(0)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "divortio-lz4_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".c", ".h")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "import oracle" not in text and "lz4_oracle" not in text and "from oracle" not in text, f


def test_frames_info_walks_concatenated_and_skippable_frames_on_the_host():
    """dlz4_frames_info is host-only (header parse + block walk): counts, bounds and errors without a GPU."""
    import struct
    import oracle
    a, b = b"frame one " * 5000, bytes(range(256)) * 3000
    fa = oracle.compress_buffer(a, None, 65536, True, True, True)
    fb = oracle.compress_buffer(b, None, 4194304, False, False, False)          # no content size: bound from the block table
    skip = struct.pack("<II", 0x184D2A5F, 5) + b"xxxxx"
    L = api.lib()

    def info(buf):
        arr = np.frombuffer(buf, dtype=np.uint8)
        total, count = C.c_uint64(0), C.c_uint32(0)
        st = L.dlz4_frames_info(arr.ctypes.data, arr.size, C.byref(total), C.byref(count))
        return st, int(total.value), int(count.value)

    st, total, count = info(skip + fa + skip + fb + skip)
    assert st == 0 and count == 2 and total >= len(a) + len(b)
    assert info(fa)[1:] == (len(a), 1)
    assert info(fa + b"\x00\x01\x02\x03")[0] == api.E_BAD_MAGIC
    assert info(fa[:-3])[0] != 0                                                  # truncated content checksum / EndMark
    assert info(struct.pack("<II", 0x184D2A50, 100) + b"short")[0] != 0          # skippable frame longer than the buffer
    fi = api.FrameInfo()
    arr = np.frombuffer(fa + fb, dtype=np.uint8)
    assert L.dlz4_frame_info(arr.ctypes.data, arr.size, C.byref(fi)) == 0 and fi.frame_bytes == len(fa)


def test_stateful_xxh32_digest_of_short_inputs_needs_no_device():
    """Below one 16-byte stripe dlz4_xxh32_update only buffers and dlz4_xxh32_digest finishes on the host (xxhash32.js:67-97)."""
    import oracle
    L = api.lib()
    for seed in (0, 7):
        for data in (b"", b"a", b"Hello World", b"123456789012345"):
            s = api.Xxh32State()
            L.dlz4_xxh32_reset(C.byref(s), seed)
            for k in range(len(data)):                                            # byte by byte: never reaches a stripe
                arr = np.frombuffer(data[k:k + 1], dtype=np.uint8)
                # ctx is only dereferenced when a stripe is ready; a dummy non-null handle is never touched here
                assert L.dlz4_xxh32_update(C.c_void_p(1), C.byref(s), arr.ctypes.data, 1) == 0
            assert L.dlz4_xxh32_digest(C.byref(s)) == oracle.xxh32(data, seed)
    assert L.dlz4_xxh32_digest(C.byref(s)) == oracle.xxh32(b"123456789012345", 7)


def test_napi_addon_type_checks_against_the_header():
    """addon/dlz4_napi.c (the binding INTEGRATION.md describes) compiles with -fsyntax-only -Wall -Wextra -Werror against
    include/dlz4_b200.h and a hand-declared Node-API subset; every C-ABI entry point it calls exists with that signature."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run(["make", "-C", os.path.join(root, "addon"), "syntax"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
