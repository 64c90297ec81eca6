"""Seek table writer (SURVEY §8f rank 4), CPU only: frames come from the oracle, the table from the product's host code,
and the reference's own seekable reader (contrib/seekable_format/zstdseek_decompress.c, compiled in place into
oracle/_ref/libzstd_seekable_ref.so; its answers are recorded under tests/golden/reference/ for machines without it) must
find every frame and decompress arbitrary ranges."""
import ctypes
import os
import random

import pytest

import zref
import zstd_b200

SEEK_SO = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libzstd_seekable_ref.so")


def _seekable_reader(blob, ranges):
    """what the reference's seekable reader reports for blob: the number of frames, each frame's compressed offset and
    a digest (zref.sha16) of each decompressed range (start, length)"""
    S = ctypes.CDLL(SEEK_SO)
    S.ZSTD_seekable_create.restype = ctypes.c_void_p
    S.ZSTD_seekable_initBuff.restype = ctypes.c_size_t
    S.ZSTD_seekable_initBuff.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
    S.ZSTD_seekable_decompress.restype = ctypes.c_size_t
    S.ZSTD_seekable_decompress.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_ulonglong]
    S.ZSTD_seekable_getNumFrames.restype = ctypes.c_uint
    S.ZSTD_seekable_getNumFrames.argtypes = [ctypes.c_void_p]
    S.ZSTD_seekable_getFrameCompressedOffset.restype = ctypes.c_ulonglong
    S.ZSTD_seekable_getFrameCompressedOffset.argtypes = [ctypes.c_void_p, ctypes.c_uint]
    S.ZSTD_seekable_free.argtypes = [ctypes.c_void_p]
    zs = S.ZSTD_seekable_create()
    r = S.ZSTD_seekable_initBuff(zs, blob, len(blob))
    assert not zref.ref().ZSTD_isError(r)
    n = S.ZSTD_seekable_getNumFrames(zs)
    offsets = [S.ZSTD_seekable_getFrameCompressedOffset(zs, i) for i in range(n)]
    digests = []
    for a, k in ranges:
        out = ctypes.create_string_buffer(k)
        got = S.ZSTD_seekable_decompress(zs, out, k, a)
        digests.append(zref.sha16(out.raw) if got == k else None)
    S.ZSTD_seekable_free(zs)
    return [n, offsets, digests]


def test_reference_reader_accepts_our_seek_table():
    rng = random.Random(5)
    sizes = [1024] * 20 + [0, 70_000, 300_000, 5, 128 << 10]
    src = zref.synthetic(sum(sizes), 9, 0.5)
    frames, off = [], 0
    for n in sizes:
        frames.append(zref.oracle_compress(src[off:off + n], 1)); off += n
    blob = b"".join(frames) + zstd_b200.seek_table([len(f) for f in frames], sizes)
    assert len(blob) == sum(len(f) for f in frames) + 17 + 8 * len(sizes)
    assert blob[-4:] == bytes.fromhex("b1ea928f")                                   # Seekable_Magic_Number, little-endian
    assert zref.ref_decodes(blob, src)                                              # the table is a skippable frame for a plain decoder
    ranges = []
    for _ in range(50):
        a = rng.randrange(0, len(src)); n = rng.randrange(1, min(100_000, len(src) - a) + 1)
        ranges.append((a, n))
    nframes, offsets, digests = zref.recorded(zref._key("seekable", blob, ranges), lambda: _seekable_reader(blob, ranges))
    assert nframes == len(sizes)
    pos = 0
    for i, f in enumerate(frames):
        assert offsets[i] == pos
        pos += len(f)
    for (a, n), h in zip(ranges, digests):
        assert h == zref.sha16(src[a:a + n]), (a, n)


def test_seek_table_errors():
    L = zstd_b200.lib()
    L.ZSTDB200_writeSeekTable.restype = ctypes.c_size_t
    L.ZSTDB200_writeSeekTable.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]
    one = (ctypes.c_size_t * 1)(10)
    dst = ctypes.create_string_buffer(64)
    r = L.ZSTDB200_writeSeekTable(dst, 24, one, one, 1)                             # needs 25 bytes
    assert L.ZSTD_isError(r) and L.ZSTD_getErrorCode(r) == 70
    big = (ctypes.c_size_t * 1)(1 << 32)
    r = L.ZSTDB200_writeSeekTable(dst, 64, big, one, 1)                             # sizes are 32-bit fields
    assert L.ZSTD_isError(r) and L.ZSTD_getErrorCode(r) == 72
    assert L.ZSTDB200_writeSeekTable(dst, 64, None, None, 0) == 17                  # empty table: header + footer
