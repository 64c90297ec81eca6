"""CPU tests of the decompressor's format-level code (zstd_b200/csrc/zb_decode_core.cuh): tests/host_decode.cpp drives the
same host+device functions the CUDA kernels call, block after block, and must reproduce the input of frames written by
the reference encoder (every level, so Huffman treeless / FSE repeat modes, RLE tables, long offsets ...), by this repo's
oracle, and of the reference's own golden decompression vectors (tests/golden/decompression*, copied from the reference's
tests/golden-decompression*).  The reference's frames and verdicts come from tests/golden/reference/ where it is not built."""
import ctypes
import glob
import os
import subprocess

import pytest

import zref

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libzb_hostdecode.so")


@pytest.fixture(scope="module")
def H():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-Wall", "-Wextra", "-Werror", "-Wno-unused-function", "-x", "c++",
                           "-o", SO, os.path.join(HERE, "host_decode.cpp")])
    h = ctypes.CDLL(SO)
    h.zbh_decompress.restype = ctypes.c_size_t
    h.zbh_decompress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
    return h


def dec(H, frame, cap):
    out = ctypes.create_string_buffer(cap + 16)
    r = H.zbh_decompress(out, cap, frame, len(frame))
    if r > (1 << 63):
        return ("ERR", (1 << 64) - r)
    return out.raw[:r]


INPUTS = {
    "empty": b"", "one": b"x", "tiny": b"hello hello hello hello", "zeros": bytes(500_000), "rand": zref.random_bytes(200_000, 1),
    "period3": b"abc" * 50_000, "syn": zref.synthetic(300_000, 9), "syn-p90": zref.synthetic(1 << 20, 6, 0.9),
}


@pytest.mark.parametrize("level", [1, 3, -3, 5, 9, 15, 19])
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_reference_frames(H, name, level):
    data = INPUTS[name]
    assert dec(H, zref.ref_frame(data, level), len(data)) == data


@pytest.mark.parametrize("level", [1, 3, -3])
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_oracle_frames(H, name, level):
    data = INPUTS[name]
    assert dec(H, zref.oracle_compress(data, level), len(data)) == data


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary not built")
@pytest.mark.parametrize("p,level", [(50, 1), (90, 3), (30, -3), (50, 7), (90, 19)])
def test_datagen_multi_block(H, p, level):
    """8 MiB: 64 blocks, tables reused across blocks (treeless literals, repeat-mode sequence tables)"""
    data = zref.datagen(8 << 20, p)
    assert dec(H, zref.ref_frame(data, level), len(data)) == data


def test_golden_inputs_all_levels(H):
    for g in ("large-literal-and-match-lengths", "http", "PR-3517-block-splitter-corruption-test", "huffman-compressed-larger"):
        data = zref.golden_input(g)
        for level in (1, 3, 6, 12, 19, -5):
            assert dec(H, zref.ref_frame(data, level), len(data)) == data, (g, level)


def test_concatenated_and_skippable_frames(H):
    a, b = b"abc" * 1000, zref.synthetic(300_000, 3)
    skip = bytes([0x53, 0x2A, 0x4D, 0x18, 5, 0, 0, 0]) + b"xxxxx"
    stream = zref.ref_frame(a, 3) + skip + zref.ref_frame(b, 1) + skip
    assert dec(H, stream, len(a) + len(b)) == a + b


def test_reference_golden_decompression_vectors(H):
    for f in sorted(glob.glob(os.path.join(zref.GOLDEN, "decompression", "*.zst"))):
        frame = open(f, "rb").read()
        got = dec(H, frame, 1 << 21)
        assert not isinstance(got, tuple), (f, got)
        assert zref.sha16(got) == zref.ref_decoded_digest(frame, 1 << 21), f
    for f in sorted(glob.glob(os.path.join(zref.GOLDEN, "decompression-errors", "*.zst"))):
        got = dec(H, open(f, "rb").read(), 1 << 21)
        assert got == ("ERR", 20), (f, got)                     # corruption_detected, as the reference reports


def test_truncated_and_garbage(H):
    data = zref.synthetic(100_000, 5)
    frame = zref.ref_frame(data, 3)
    assert dec(H, frame[:-1], len(data))[0] == "ERR"
    assert dec(H, frame[: len(frame) // 2], len(data))[0] == "ERR"
    assert dec(H, b"\x00\x01\x02\x03\x04\x05\x06\x07", 100) == ("ERR", 10)          # prefix_unknown
    assert dec(H, frame, len(data) - 1) == ("ERR", 70)                              # dstSize_tooSmall


@pytest.mark.parametrize("kind", ["zdict", "raw"])
def test_dictionaries(H, kind):
    d = zref.golden_input("zdict-16k-synthetic-seed77") if kind == "zdict" else zref.synthetic(20_000, 5, 0.5)
    H.zbh_decompress_usingDict.restype = ctypes.c_size_t
    H.zbh_decompress_usingDict.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]

    def dd(frame, n):
        out = ctypes.create_string_buffer(n + 16)
        r = H.zbh_decompress_usingDict(out, n, frame, len(frame), d, len(d))
        return ("ERR", (1 << 64) - r) if r > (1 << 63) else out.raw[:r]
    for n in (0, 1, 100, 1000, 5000, 200_000):
        src = zref.synthetic(n, 31, 0.5) if n else b""
        for level in (1, 3, -3, 6, 19):
            assert dd(zref.ref_frame(src, level, d), n) == src, (n, level)
        for level in (1, 3):
            assert dd(zref.oracle_compress_using_dict(src, d, level), n) == src, (n, level)
    recs = [zref.synthetic(1024, 100 + i, 0.5) for i in range(50)]
    assert dd(b"".join(zref.ref_frame(r, 1, d) for r in recs), 50 * 1024) == b"".join(recs)


def test_corrupted_frames_differential(H):
    """bit flips in valid frames (both encoders): the decoder's format code never reads out of bounds (the same functions
    run under ASAN / UBSAN in development: 6000 runs clean) and never accepts what the reference decoder refuses; when both
    accept, the bytes agree.  (The reference accepts some Huffman streams that over-read their start; here that is
    corruption_detected.)"""
    import random
    rng = random.Random(99)
    srcs = [zref.synthetic(n, s, p) for n, s, p in ((300, 1, 0.5), (5000, 2, 0.7), (70_000, 3, 0.5), (200_000, 4, 0.9))] + [b"abc" * 20_000]
    frames = []
    for s in srcs:
        for level in (1, 3, 19):
            frames.append((zref.ref_frame(s, level), len(s)))
        frames.append((zref.oracle_compress(s, 1), len(s)))
    both = 0
    for _ in range(800):
        f, size = rng.choice(frames)
        b = bytearray(f)
        for _ in range(rng.choice((1, 1, 2))):
            b[rng.randrange(len(b))] ^= 1 << rng.randrange(8)
        cap = size + 32
        ours = dec(H, bytes(b), cap)
        ref = zref.ref_decoded_digest(bytes(b), cap)
        if not isinstance(ours, tuple):
            assert ref is not None and zref.sha16(ours) == ref
            both += 1
    assert both > 100
