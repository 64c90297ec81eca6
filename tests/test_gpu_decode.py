"""GPU decompression (pytest -m gpu): ZSTD_decompress / ZSTD_decompressDCtx / ZSTDB200_decompressDevice through the C ABI
must reproduce the input of this library's own frames and of the reference encoder's frames (every level), and must
agree with the reference decoder on the reference's golden vectors.  The reference's frames and verdicts come from
tests/golden/reference/ where it is not built."""
import ctypes
import glob
import os

import pytest

import zref
import zstd_b200
from test_gpu_parity import CASES

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600, method="thread")]      # a stuck kernel must fail the run, not hang it


@pytest.fixture(scope="module")
def cctx():
    c = zstd_b200.ZSTD_CCtx()
    yield c
    c.close()


@pytest.fixture(scope="module")
def dctx():
    d = zstd_b200.ZSTD_DCtx()
    yield d
    d.close()


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("level", [1, 3, -3])
def test_round_trip_of_own_frames(cctx, dctx, name, level):
    src = CASES[name]
    assert dctx.decompress(cctx.compress(src, level), len(src)) == src


@pytest.mark.parametrize("name", ["empty", "one", "tiny-rep", "zeros-1M", "rand-300k", "period3", "syn-70000", "syn-400000", "syn-4M-p30", "syn-4M-p90", "syn-2M-p10"])
@pytest.mark.parametrize("level", [1, 3, -5, 6, 12, 19])
def test_reference_frames(dctx, name, level):
    src = CASES[name]
    assert dctx.decompress(zref.ref_frame(src, level), len(src)) == src


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary not built")
@pytest.mark.parametrize("p,level", [(50, 1), (90, 3), (30, -3), (50, 9)])
def test_datagen_64MiB(cctx, dctx, p, level):
    src = zref.datagen(64 << 20, p)
    assert dctx.decompress(zref.ref_frame(src, level), len(src)) == src
    if level < 5:
        assert dctx.decompress(cctx.compress(src, level), len(src)) == src


def test_concatenated_skippable_and_checksum(dctx):
    a, b = b"abc" * 1000, zref.synthetic(300_000, 3)
    skip = bytes([0x53, 0x2A, 0x4D, 0x18, 5, 0, 0, 0]) + b"xxxxx"
    stream = zref.ref_frame(a, 3) + skip + zref.ref_frame(b, 1) + skip
    assert dctx.decompress(stream, len(a) + len(b)) == a + b
    # a frame with a content checksum (written by this library's ZSTD_compress2): verified, and a flipped bit is noticed
    c = zstd_b200.ZSTD_CCtx()
    c.set_parameter("checksum_flag", 1)
    f = bytearray(c.compress2(b))
    c.close()
    assert dctx.decompress(bytes(f), len(b)) == b
    f[-1] ^= 1
    with pytest.raises(zstd_b200.ZstdError) as e:
        dctx.decompress(bytes(f), len(b))
    assert e.value.code == 22


def test_golden_decompression_vectors(dctx):
    for f in sorted(glob.glob(os.path.join(zref.GOLDEN, "decompression", "*.zst"))):
        frame = open(f, "rb").read()
        got = dctx.decompress(frame, 1 << 21)
        assert zref.sha16(got) == zref.ref_decoded_digest(frame, 1 << 21), f
    for f in sorted(glob.glob(os.path.join(zref.GOLDEN, "decompression-errors", "*.zst"))):
        with pytest.raises(zstd_b200.ZstdError) as e:
            dctx.decompress(open(f, "rb").read(), 1 << 21)
        assert e.value.code == 20, f


def test_errors(cctx, dctx):
    src = zref.synthetic(100_000, 5)
    frame = cctx.compress(src, 1)
    for bad, code in ((frame[:-1], None), (frame[: len(frame) // 2], None), (b"\x00\x01\x02\x03\x04\x05\x06\x07", 10)):
        with pytest.raises(zstd_b200.ZstdError) as e:
            dctx.decompress(bad, len(src))
        assert code is None or e.value.code == code
    with pytest.raises(zstd_b200.ZstdError) as e:
        dctx.decompress(frame, len(src) - 1)
    assert e.value.code == 70
    assert zstd_b200.lib().ZSTD_getFrameContentSize(frame, len(frame)) == len(src)
    assert zstd_b200.lib().ZSTD_findFrameCompressedSize(frame, len(frame)) == len(frame)
    assert zstd_b200.ZSTD_decompress(frame) == src


def test_device_buffers(cctx, dctx):
    import torch
    src = zref.synthetic(9 << 20, 21, 0.5)
    frames = cctx.compress(src[: 5 << 20], 1) + cctx.compress(src[5 << 20:], 3)
    d_in = torch.frombuffer(bytearray(frames), dtype=torch.uint8).cuda()
    d_out = torch.empty(len(src), dtype=torch.uint8, device="cuda")
    n = dctx.decompress_device(d_out.data_ptr(), len(src), d_in.data_ptr(), len(frames))
    assert n == len(src) and bytes(d_out.cpu().numpy()) == src
    st = dctx.stats()
    assert st.nbFrames == 2 and st.nbBlocks == 72
    # the same through the kernel walk (inputs beyond 512 MiB take it; forced here)
    os.environ["ZSTDB200_HOSTWALK_MAX"] = "0"
    try:
        d2 = zstd_b200.ZSTD_DCtx()
    finally:
        del os.environ["ZSTDB200_HOSTWALK_MAX"]
    d_out.zero_()
    assert d2.decompress_device(d_out.data_ptr(), len(src), d_in.data_ptr(), len(frames)) == len(src)
    assert bytes(d_out.cpu().numpy()) == src
    d2.close()


@pytest.mark.parametrize("kind", ["zdict", "raw"])
def test_dictionaries(cctx, dctx, kind):
    """ZSTD_decompress_usingDict: frames written with a dictionary by the reference (every level) and by this library"""
    d = zref.golden_input("zdict-16k-synthetic-seed77") if kind == "zdict" else zref.synthetic(20_000, 5, 0.5)
    L = zstd_b200.lib()
    L.ZSTD_decompress_usingDict.restype = ctypes.c_size_t
    L.ZSTD_decompress_usingDict.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]

    def dec(frames, n):
        out = ctypes.create_string_buffer(max(n, 1))
        r = L.ZSTD_decompress_usingDict(dctx._h, out, n, frames, len(frames), d, len(d))
        assert not L.ZSTD_isError(r), L.ZSTD_getErrorName(r)
        return out.raw[:r]
    for n in (0, 1, 100, 1000, 5000, 200_000):
        src = zref.synthetic(n, 31, 0.5) if n else b""
        for level in (1, 3, -3, 6, 19):
            assert dec(zref.ref_frame(src, level, d), n) == src, (n, level)
        for level in (1, 3):
            assert dec(cctx.compress_using_dict(src, d, level), n) == src, (n, level)
    # config 5 in miniature: many records, one call
    recs = [zref.synthetic(1024, 100 + i, 0.5) for i in range(300)]
    stream = b"".join(zref.ref_frame(r, 1, d) for r in recs)
    assert dec(stream, 300 * 1024) == b"".join(recs)
    if kind == "zdict":                                        # a frame that names another dictionary
        other = bytearray(d); other[4] ^= 1
        out = ctypes.create_string_buffer(2048)
        r = L.ZSTD_decompress_usingDict(dctx._h, out, 2048, stream[:200], 200, bytes(other), len(other))
        assert L.ZSTD_isError(r)


def test_streaming_decompression(cctx):
    """ZSTD_decompressStream: input arriving in arbitrary pieces, output handed out through a small buffer; frames of both
    encoders, several frames in one stream"""
    L = zstd_b200.lib()

    class Buf(ctypes.Structure):
        _fields_ = [("p", ctypes.c_void_p), ("size", ctypes.c_size_t), ("pos", ctypes.c_size_t)]
    L.ZSTD_createDStream.restype = ctypes.c_void_p
    L.ZSTD_freeDStream.argtypes = [ctypes.c_void_p]
    L.ZSTD_initDStream.restype = ctypes.c_size_t; L.ZSTD_initDStream.argtypes = [ctypes.c_void_p]
    L.ZSTD_decompressStream.restype = ctypes.c_size_t; L.ZSTD_decompressStream.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    a, b = zref.synthetic(300_000, 41, 0.5), zref.synthetic(70_001, 42, 0.7)
    stream = cctx.compress(a, 1) + (zref.ref_compress(b, 5) if zref.have_ref() else cctx.compress(b, 3)) + cctx.compress(b"", 1)
    zds = L.ZSTD_createDStream()
    assert not L.ZSTD_isError(L.ZSTD_initDStream(zds))
    out = bytearray()
    room = ctypes.create_string_buffer(10_000)
    pos, last = 0, None
    for piece in (1, 7, 100, 50_000, 3, len(stream)):
        chunk = stream[pos:pos + piece]; pos += len(chunk)
        sbuf = ctypes.create_string_buffer(chunk, max(len(chunk), 1))
        i = Buf(ctypes.cast(sbuf, ctypes.c_void_p), len(chunk), 0)
        for _ in range(10_000):
            o = Buf(ctypes.cast(room, ctypes.c_void_p), len(room), 0)
            last = L.ZSTD_decompressStream(zds, ctypes.byref(o), ctypes.byref(i))
            assert not L.ZSTD_isError(last), L.ZSTD_getErrorName(last)
            out += room.raw[:o.pos]
            if i.pos == i.size and o.pos < len(room):
                break
    assert last == 0 and bytes(out) == a + b
    L.ZSTD_freeDStream(zds)
