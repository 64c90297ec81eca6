"""GPU parity tests (run on the B200 box: pytest -m gpu).  Every call goes through the C ABI of
libzstd_b200.so.  The CUDA path must be bit-exact with the oracle, every frame must decode with the
reference decoder, sizes must stay within the two-sided bound of zref.size_delta_ok of the reference's (the north
star's 0.5 % is met on part of the grid only: DESIGN.md section 5).  The reference's answers come from the compiled
library where it is built and from tests/golden/reference/ elsewhere."""
import ctypes
import json
import os

import pytest

import zref
import zstd_b200

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = zstd_b200.ZSTD_CCtx()
    yield c
    c.close()


def decode_ok(frame, src):
    assert zref.ref_decodes(frame, src)


CASES = {
    "empty": b"", "one": b"x", "six": b"abcdef", "seven": b"abcdefg", "tiny-rep": b"abcabcabc" * 10,
    "zeros-300": bytes(300), "zeros-1M": bytes(1 << 20), "zeros-128k+1": bytes((128 << 10) + 1),
    "rand-100k": zref.random_bytes(100_000, 1), "rand-300k": zref.random_bytes(300_000, 2),
    "period3": b"abc" * 50_000, "period40": bytes(range(40)) * 9000,
    "syn-100": zref.synthetic(100, 100), "syn-1000": zref.synthetic(1000, 1000), "syn-5000": zref.synthetic(5000, 5000),
    "syn-70000": zref.synthetic(70_000, 7), "syn-128k": zref.synthetic(128 << 10, 3), "syn-128k+1": zref.synthetic((128 << 10) + 1, 3),
    "syn-400000": zref.synthetic(400_000, 4), "syn-4M-p30": zref.synthetic(4 << 20, 5, 0.3), "syn-4M-p90": zref.synthetic(4 << 20, 6, 0.9),
    "syn-2M-p10": zref.synthetic(2 << 20, 8, 0.1),
}
# sizes around the 16 KiB parse-segment boundaries, and matches that want to cross every segment end
SEG = 16 << 10
for _n in (SEG - 1, SEG, SEG + 1, SEG + 6, SEG + 7, SEG + 8, 2 * SEG + 3, 8 * SEG - 1, 8 * SEG + SEG + 5, 3 * 8 * SEG + 9):
    CASES[f"seg-{_n}"] = zref.synthetic(_n, 40 + _n % 7, 0.6)
CASES["seg-rep"] = (zref.synthetic(5000, 77, 0.3) * 30)[: 9 * SEG + 123]
CASES["seg-zeros"] = bytes(5 * SEG + 11)


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("level", [1, 2, 3, -1, -3, -7])
def test_bit_exact_with_oracle(ctx, name, level):
    src = CASES[name]
    got = ctx.compress(src, level)
    assert got == zref.oracle_compress(src, level)
    decode_ok(got, src)


def test_simple_api_temporary_context():
    """ZSTD_compress (lib/zstd.h:155) creates and frees its own context."""
    src = zref.synthetic(300_000, 11)
    assert zstd_b200.ZSTD_compress(src, 1) == zref.oracle_compress(src, 1)


def test_context_reuse_and_determinism(ctx):
    """fuzzer.c:1547-1589 "re-using a CCtx should compress the same"; fuzz/simple_round_trip.c determinism."""
    a = zref.synthetic(1 << 20, 21)
    b = zref.synthetic(200_000, 22, 0.8)
    fa1 = ctx.compress(a, 1)
    fb = ctx.compress(b, -3)
    fa2 = ctx.compress(a, 1)
    assert fa1 == fa2
    c2 = zstd_b200.ZSTD_CCtx()
    assert c2.compress(a, 1) == fa1 and c2.compress(b, -3) == fb
    c2.close()


def test_dst_too_small(ctx):
    """fuzzer.c:4550-4562: too small a destination returns dstSize_tooSmall and never writes past it."""
    src = zref.synthetic(300_000, 1)
    full = ctx.compress(src, 1)
    L = zstd_b200.lib()
    for cap in (5, 17, 18, 100, len(full) - 1):
        dst = ctypes.create_string_buffer(cap + 64)
        ctypes.memset(dst, 0xA5, cap + 64)
        r = L.ZSTD_compressCCtx(ctx._h, dst, cap, src, len(src), 1)
        assert L.ZSTD_isError(r) and L.ZSTD_getErrorCode(r) == 70
        assert dst.raw[cap:] == b"\xa5" * 64
    dst = ctypes.create_string_buffer(len(full))
    assert L.ZSTD_compressCCtx(ctx._h, dst, len(full), src, len(src), 1) == len(full)
    assert dst.raw == full


def test_golden_inputs(ctx):
    """The reference's tests/golden-compression inputs through our entry points (cli-tests/compression/golden.sh)."""
    frames = json.load(open(os.path.join(zref.GOLDEN, "frames.json")))
    for key, rec in frames.items():
        name, level = key.rsplit("@", 1)
        path = os.path.join(zref.GOLDEN, "inputs", name)
        if not os.path.exists(path):
            continue
        data = open(path, "rb").read()
        out = ctx.compress(data, int(level))
        assert len(out) == rec["oracle_size"] and zref.sha(out) == rec["oracle_sha256"], key
        assert zref.size_delta_ok(len(out), rec["ref_size"], len(data)), (key, len(out), rec["ref_size"])      # against the REFERENCE's size
        decode_ok(out, data)


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary absent")
@pytest.mark.parametrize("p,level,size", [(50, 1, 16 << 20), (30, -3, 64 << 20), (90, 3, 64 << 20)])
def test_baseline_configs_size_and_roundtrip(ctx, p, level, size):
    """configs[0] (datagen -g16MB -P50, level 1), 64 MiB samples of config 3 (P30, --fast=3) and config 4 (P90, level 3):
    bit-exact with the oracle, decodes, size within +-0.5 % of the reference."""
    src = zref.datagen(size, p)
    got = ctx.compress(src, level)
    assert got == zref.oracle_compress(src, level)
    decode_ok(got, src)
    ref = zref.ref_size(src, level)
    delta = (len(got) - ref) / ref
    assert zref.size_delta_ok(len(got), ref, len(src)), f"{delta:+.4%}"


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary absent")
@pytest.mark.parametrize("size", [1 << 20, 64 << 20])
@pytest.mark.parametrize("level", [1, 3, -3])
@pytest.mark.parametrize("p", [30, 50, 90])
def test_size_vs_reference_grid(ctx, p, level, size):
    """datagen P30 / P50 / P90 x levels 1 / 3 / -3 x 1 MiB / 64 MiB: one insertion rule and one table shape per level
    class must serve all of them (round 1 fitted level 3 to P90 alone).  GPU bytes == oracle bytes, the reference
    decodes them, and the size stays inside the two-sided bound of zref.size_delta_ok (measured values: DESIGN.md 5)."""
    src = zref.datagen(size, p)
    got = ctx.compress(src, level)
    if size <= (1 << 20):
        assert got == zref.oracle_compress(src, level)
    decode_ok(got, src)
    ref = zref.ref_size(src, level)
    assert zref.size_delta_ok(len(got), ref, len(src)), f"{(len(got) - ref) / ref:+.4%}"


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary absent")
def test_full_size_config2_properties(ctx):
    """configs[1] at full size (datagen -g1GB -P50, level 1), device-resident.  The oracle would need
    ~10 s here, so this checks size-independent properties: the frame decodes to the input, the
    run is deterministic, and cutting the same bytes into 64 MiB frames decodes to the same bytes."""
    import torch
    size = 1 << 30
    src = zref.datagen(size, 50)
    d_src = torch.frombuffer(bytearray(src), dtype=torch.uint8).cuda()
    cap = zstd_b200.ZSTD_compressBound(size) + 64 * 32
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    n1 = ctx.compress_device(d_dst.data_ptr(), cap, d_src.data_ptr(), size, 1)
    f1 = bytes(d_dst[:n1].cpu().numpy())
    n2 = ctx.compress_device(d_dst.data_ptr(), cap, d_src.data_ptr(), size, 1)
    assert n1 == n2 and bytes(d_dst[:n2].cpu().numpy()) == f1
    decode_ok(f1, src)
    fs = 64 << 20
    offs = list(range(0, size, fs))
    total, csz = ctx.compress_frames(d_dst.data_ptr(), cap, d_src.data_ptr(), offs, [fs] * len(offs), level=1, device_memory=True)
    assert sum(csz) == total
    decode_ok(bytes(d_dst[:total].cpu().numpy()), src)          # concatenated frames, lib/zstd.h:160-162
    ref = zref.ref_size(src[: 256 << 20], 1)
    part = ctx.compress(src[: 256 << 20], 1)
    assert zref.size_delta_ok(len(part), ref, 256 << 20)


def test_many_small_frames(ctx):
    """Independent small frames in one call (shape of config 5 without the dictionary)."""
    import torch
    rec = 1024
    n = 2048
    src = zref.synthetic(rec * n, 33, 0.5)
    d_src = torch.frombuffer(bytearray(src), dtype=torch.uint8).cuda()
    cap = sum(zstd_b200.ZSTD_compressBound(rec) + 32 for _ in range(n))
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    total, csz = ctx.compress_frames(d_dst.data_ptr(), cap, d_src.data_ptr(), [i * rec for i in range(n)], [rec] * n, level=1)
    out = bytes(d_dst[:total].cpu().numpy())
    pos = 0
    for i in range(0, n, 97):
        start = sum(csz[:i])
        assert out[start:start + csz[i]] == zref.oracle_compress(src[i * rec:(i + 1) * rec], 1)
    decode_ok(out, src)


@pytest.mark.parametrize("dict_name", ["zdict-16k-synthetic-seed77", "http-dict-missing-symbols", "zero-weight-dict", "raw-32k"])
def test_compress_using_dict(ctx, dict_name):
    """ZSTD_compress_usingDict (lib/zstd.h:944), config-5 shape: 1 KiB records + shared dictionary; also
    empty / tiny / multi-block inputs.  Bit-exact with the oracle, decodable by ZSTD_decompress_usingDict."""
    d = zref.synthetic(32 << 10, 123, 0.5) if dict_name == "raw-32k" else zref.golden_input(dict_name)
    data = zref.synthetic(1024 * 64, 5, 0.5)
    srcs = [data[i * 1024:(i + 1) * 1024] for i in range(64)] + [b"", b"a", d[-2000:-900], zref.golden_input("http"), zref.synthetic(300_000, 8)]
    for src in srcs:
        got = ctx.compress_using_dict(src, d, 1)
        assert got == zref.oracle_compress_using_dict(src, d, 1)
        assert zref.ref_decodes(got, src, d)
    assert ctx.compress_using_dict(srcs[0], b"1234567", 1) == ctx.compress(srcs[0], 1)        # < 8 bytes: ignored


def test_many_records_with_dictionary(ctx):
    """BASELINE config 5 in one call: N x 1 KiB records + one shared dictionary -> N frames."""
    import torch
    d = zref.golden_input("zdict-16k-synthetic-seed77")
    rec, n = 1024, 4096
    src = zref.synthetic(rec * n, 91, 0.5)
    d_src = torch.frombuffer(bytearray(src), dtype=torch.uint8).cuda()
    cap = n * (zstd_b200.ZSTD_compressBound(rec) + 32)
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    total, csz = ctx.compress_frames(d_dst.data_ptr(), cap, d_src.data_ptr(), [i * rec for i in range(n)], [rec] * n, level=1, dict_bytes=d)
    out = bytes(d_dst[:total].cpu().numpy())
    assert sum(csz) == total
    pos = 0
    for i in range(n):
        if i % 131 == 0:
            assert out[pos:pos + csz[i]] == zref.oracle_compress_using_dict(src[i * rec:(i + 1) * rec], d, 1)
            assert zref.ref_decodes(out[pos:pos + csz[i]], src[i * rec:(i + 1) * rec], d)
        pos += csz[i]


@pytest.mark.parametrize("level", [1, 3, -3])
@pytest.mark.parametrize("dict_name", ["zdict-16k-synthetic-seed77", "raw-32k"])
def test_compress_using_cdict(ctx, dict_name, level):
    """ZSTD_createCDict / ZSTD_compress_usingCDict (lib/zstd.h:967-995; SURVEY.md §8f rank 1): same bytes as
    ZSTD_compress_usingDict at the CDict's level = the oracle's, decodable by the reference, stable across
    repeated calls and across contexts sharing the CDict."""
    d = zref.synthetic(32 << 10, 123, 0.5) if dict_name == "raw-32k" else zref.golden_input(dict_name)
    data = zref.synthetic(1024 * 48, 15, 0.5)
    srcs = [data[i * 1024:(i + 1) * 1024] for i in range(48)] + [b"", b"a", d[-2000:-900], zref.synthetic(300_000, 8)]
    cd = zstd_b200.ZSTD_CDict(d, level)
    ctx2 = zstd_b200.ZSTD_CCtx()
    assert cd.dict_id == (zstd_b200.lib().ZSTD_getDictID_fromDict(d, len(d)))
    assert (cd.dict_id != 0) == (dict_name != "raw-32k")
    for k, src in enumerate(srcs):
        got = (ctx if k % 2 else ctx2).compress_using_cdict(src, cd)
        assert got == zref.oracle_compress_using_dict(src, d, level)
        if k < 4:
            assert got == ctx.compress_using_dict(src, d, level)
            assert got == ctx.compress_using_cdict(src, cd)
        assert zref.ref_decodes(got, src, d)
    ctx2.close()
    cd.close()


def test_many_records_with_cdict(ctx):
    """Config 5 through the digested dictionary: one batch call, host and device buffers, equals per-record calls."""
    import torch
    d = zref.golden_input("zdict-16k-synthetic-seed77")
    rec, n = 1024, 2048
    src = zref.synthetic(rec * n, 92, 0.5)
    cd = zstd_b200.ZSTD_CDict(d, 1)
    d_src = torch.frombuffer(bytearray(src), dtype=torch.uint8).cuda()
    cap = n * (zstd_b200.ZSTD_compressBound(rec) + 32)
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    offs, sizes = [i * rec for i in range(n)], [rec] * n
    for rep in range(2):                                  # second call reuses the cached table image
        total, csz = ctx.compress_frames_using_cdict(d_dst.data_ptr(), cap, d_src.data_ptr(), offs, sizes, cd)
        out = bytes(d_dst[:total].cpu().numpy())
        assert sum(csz) == total
        pos = 0
        for i in range(n):
            if i % 97 == 0:
                assert out[pos:pos + csz[i]] == zref.oracle_compress_using_dict(src[i * rec:(i + 1) * rec], d, 1)
            pos += csz[i]
    total2, csz2 = ctx.compress_frames(d_dst.data_ptr(), cap, d_src.data_ptr(), offs, sizes, level=1, dict_bytes=d)
    assert (total2, csz2) == (total, csz) and bytes(d_dst[:total2].cpu().numpy()) == out
    cd.close()


def test_cdict_errors():
    bad = bytearray(zref.golden_input("zdict-16k-synthetic-seed77")); bad[12:40] = b"\xff" * 28      # entropy tables destroyed
    with pytest.raises(zstd_b200.ZstdError):
        zstd_b200.ZSTD_CDict(bytes(bad), 1)
    L = zstd_b200.lib()
    c = zstd_b200.ZSTD_CCtx()
    import ctypes
    dst = ctypes.create_string_buffer(64)
    r = L.ZSTD_compress_usingCDict(c._h, dst, 64, b"abc", 3, None)
    assert L.ZSTD_isError(r) and L.ZSTD_getErrorCode(r) == 32           # dictionary_wrong, zstd_compress.c:5753
    assert L.ZSTD_freeCDict(None) == 0
    c.close()


def _with_checksum(frame: bytes, src: bytes) -> bytes:
    """What a checksummed frame must be, given the same frame without checksum: Content_Checksum_flag set in the frame
    header descriptor and the low 32 bits of XXH64(content, 0) behind the last block (zstd_compress.c:4629, :5297-5303);
    XXH64 taken from the compiled reference (ZSTD_XXH64, lib/common/xxhash.h)."""
    def xxh64():
        R = zref.ref()
        R.ZSTD_XXH64.restype = ctypes.c_ulonglong
        R.ZSTD_XXH64.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_ulonglong]
        return R.ZSTD_XXH64(src, len(src), 0)
    h = zref.recorded(zref._key("ZSTD_XXH64", src), xxh64) & 0xFFFFFFFF
    return frame[:4] + bytes([frame[4] | 4]) + frame[5:] + h.to_bytes(4, "little")


@pytest.mark.parametrize("name", ["empty", "seven", "syn-5000", "syn-128k+1", "syn-400000", "seg-rep", "rand-100k"])
def test_compress2_parameters_and_checksum(name):
    """ZSTD_CCtx_setParameter + ZSTD_compress2 (lib/zstd.h:337-603): level and checksum parameters are sticky, the frame
    equals the simple API's frame (plus flag and XXH64 word when the checksum is on), the reference decoder accepts it
    (it verifies the checksum), unsupported parameters answer parameter_unsupported."""
    src = CASES[name]
    c = zstd_b200.ZSTD_CCtx()
    for level in (1, -3, 3):
        c.set_parameter("compression_level", level)
        plain = c.compress2(src)
        assert plain == zref.oracle_compress(src, level)
        c.set_parameter("checksum_flag", 1)
        c.set_parameter("nb_workers", 4)                       # accepted, ignored
        got = c.compress2(src)
        assert got == _with_checksum(plain, src)
        assert zref.ref_decodes(got, src)
        assert got == c.compress2(src)                         # sticky + deterministic
        c.reset(2)                                              # parameters back to defaults (level 3, no checksum)
        assert c.compress2(src) == zref.oracle_compress(src, 3)
    with pytest.raises(zstd_b200.ZstdError) as e:
        c.set_parameter(101, 20)                                # ZSTD_c_windowLog
    assert e.value.code == 40
    c.close()


def test_compress2_dictionaries_and_stream2_oneshot(ctx):
    d = zref.golden_input("zdict-16k-synthetic-seed77")
    src = zref.synthetic(3000, 31, 0.5)
    c = zstd_b200.ZSTD_CCtx()
    c.set_parameter("compression_level", 1)
    c.load_dictionary(d)                                        # ZSTD_CCtx_loadDictionary: sticky
    want = zref.oracle_compress_using_dict(src, d, 1)
    assert c.compress2(src) == want and c.compress2(src) == want
    c.set_parameter("dict_id_flag", 0)                          # same frame without the dictID field
    got = c.compress2(src)
    assert (got[4] & 3) == 0 and len(got) < len(want)
    assert zref.ref_decodes(got, src, d)
    c.set_parameter("dict_id_flag", 1)
    c.load_dictionary(None)
    assert c.compress2(src) == zref.oracle_compress(src, 1)
    cd = zstd_b200.ZSTD_CDict(d, -3)
    c.ref_cdict(cd)                                             # the CDict's level applies (zstd_compress.c:5836)
    assert c.compress2(src) == zref.oracle_compress_using_dict(src, d, -3)
    c.ref_cdict(None)
    # ZSTD_compressStream2, one-shot form (lib/zstd.h:787)
    L = zstd_b200.lib()

    class Buf(ctypes.Structure):
        _fields_ = [("p", ctypes.c_void_p), ("size", ctypes.c_size_t), ("pos", ctypes.c_size_t)]
    cap = zstd_b200.ZSTD_compressBound(len(src))
    dst = ctypes.create_string_buffer(cap)
    sbuf = ctypes.create_string_buffer(src, len(src))
    o = Buf(ctypes.cast(dst, ctypes.c_void_p), cap, 0); i = Buf(ctypes.cast(sbuf, ctypes.c_void_p), len(src), 0)
    r = L.ZSTD_compressStream2(c._h, ctypes.byref(o), ctypes.byref(i), 2)
    assert r == 0 and i.pos == len(src) and dst.raw[:o.pos] == zref.oracle_compress(src, 1)
    cd.close(); c.close()


def _stream(c, chunks, directives, out_room):
    """drive ZSTD_compressStream2 the way an application does: feed chunks[i] with directives[i], draining into buffers of
    out_room bytes until the call reports completion; returns everything that came out"""
    L = zstd_b200.lib()

    class Buf(ctypes.Structure):
        _fields_ = [("p", ctypes.c_void_p), ("size", ctypes.c_size_t), ("pos", ctypes.c_size_t)]
    out = bytearray()
    dst = ctypes.create_string_buffer(out_room)
    for chunk, d in zip(chunks, directives):
        sbuf = ctypes.create_string_buffer(chunk, max(len(chunk), 1))
        i = Buf(ctypes.cast(sbuf, ctypes.c_void_p), len(chunk), 0)
        for _ in range(100000):
            o = Buf(ctypes.cast(dst, ctypes.c_void_p), out_room, 0)
            r = L.ZSTD_compressStream2(c._h, ctypes.byref(o), ctypes.byref(i), d)
            assert not L.ZSTD_isError(r), L.ZSTD_getErrorName(r)
            out += dst.raw[:o.pos]
            if i.pos == i.size and (d == 0 or r == 0):
                break
        else:
            raise AssertionError("stream made no progress")
    return bytes(out)


def test_streaming_continue_flush_end():
    """ZSTD_compressStream2 with ZSTD_e_continue / ZSTD_e_flush / ZSTD_e_end (lib/zstd.h:681-803): the output is a sequence of
    frames whose contents concatenate to the input; each flush makes everything given so far decodable"""
    src = zref.synthetic(700_000, 77, 0.5)
    c = zstd_b200.ZSTD_CCtx()
    c.set_parameter("compression_level", 1)
    parts = [src[:100_000], src[100_000:100_001], src[100_001:450_000], b"", src[450_000:]]
    # everything buffered, one frame at the end
    got = _stream(c, parts, [0, 0, 0, 0, 2], out_room=1 << 20)
    assert got == zref.oracle_compress(src, 1)
    # a flush in the middle: two frames; small output buffers: the frames trickle out
    got = _stream(c, parts, [0, 1, 0, 0, 2], out_room=4096)
    assert got == zref.oracle_compress(src[:100_001], 1) + zref.oracle_compress(src[100_001:], 1)
    assert zref.ref_decodes(got, src)
    # an empty session is an empty frame; the context is reusable afterwards
    assert _stream(c, [b""], [2], out_room=64) == zref.oracle_compress(b"", 1)
    # the older entry points
    L = zstd_b200.lib()
    L.ZSTD_initCStream.restype = ctypes.c_size_t; L.ZSTD_initCStream.argtypes = [ctypes.c_void_p, ctypes.c_int]
    assert L.ZSTD_initCStream(c._h, -3) == 0
    assert _stream(c, [src[:5000], b""], [0, 2], out_room=1 << 16) == zref.oracle_compress(src[:5000], -3)
    c.close()


def test_checksums_device_buffers_and_many_frames(ctx):
    """ZSTD_c_checksumFlag for device buffers (hashed by a warp per frame on the device) and for batch calls (host threads
    for host buffers): every frame carries the XXH64 low word the reference decoder verifies"""
    import torch
    sizes = [0, 1, 31, 32, 33, 1000, 4096, 70_000, 300_001, 7]
    src = zref.synthetic(sum(sizes), 5, 0.5)
    offs, o = [], 0
    for n in sizes:
        offs.append(o); o += n
    c = zstd_b200.ZSTD_CCtx()
    c.set_parameter("checksum_flag", 1)
    d_src = torch.frombuffer(bytearray(src), dtype=torch.uint8).cuda()
    cap = sum(zstd_b200.ZSTD_compressBound(n) + 32 for n in sizes)
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    total, csz = c.compress_frames(d_dst.data_ptr(), cap, d_src.data_ptr(), offs, sizes, level=1)
    dev = bytes(d_dst[:total].cpu().numpy())
    h_dst = ctypes.create_string_buffer(cap)
    sbuf = ctypes.create_string_buffer(src, len(src))
    total_h, csz_h = c.compress_frames(ctypes.addressof(h_dst), cap, ctypes.addressof(sbuf), offs, sizes, level=1, device_memory=False)
    assert h_dst.raw[:total_h] == dev and csz == csz_h
    pos = 0
    for off, n, k in zip(offs, sizes, csz):
        frame = dev[pos:pos + k]
        assert frame == _with_checksum(zref.oracle_compress(src[off:off + n], 1), src[off:off + n])
        pos += k
    assert zref.ref_decodes(dev, src)                          # the reference decoder checks every checksum
    # a big single frame in device memory goes through the wave executor
    big = zref.synthetic(300 << 20, 9, 0.5) if os.environ.get("ZB_BIG_TESTS") else zref.synthetic(3 << 20, 9, 0.5)
    d_big = torch.frombuffer(bytearray(big), dtype=torch.uint8).cuda()
    capb = zstd_b200.ZSTD_compressBound(len(big)) + 8
    d_out = torch.empty(capb, dtype=torch.uint8, device="cuda")
    n = c.compress_device(d_out.data_ptr(), capb, d_big.data_ptr(), len(big), level=1)
    assert bytes(d_out[:n].cpu().numpy()) == _with_checksum(zref.oracle_compress(big, 1), big)
    c.close()


def test_mixed_frame_lists(ctx):
    """Batch call over runs of equal single-block frames (the planner's template path), odd sizes, empty frames and a
    multi-block frame in between: every frame equals the single-call frame."""
    import torch
    sizes = [1024] * 50 + [5000] + [1024] * 3 + [0, 0] + [200_000] + [1024] * 10 + [7, 6, 6, 131072, 131072, 131073]
    src = zref.synthetic(sum(sizes) + 16, 123, 0.5)
    offs, o = [], 0
    for n in sizes:
        offs.append(o); o += n
    d_src = torch.frombuffer(bytearray(src), dtype=torch.uint8).cuda()
    cap = sum(zstd_b200.ZSTD_compressBound(n) + 32 for n in sizes)
    d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    total, csz = ctx.compress_frames(d_dst.data_ptr(), cap, d_src.data_ptr(), offs, sizes, level=1)
    out = bytes(d_dst[:total].cpu().numpy())
    pos = 0
    for off, n, c in zip(offs, sizes, csz):
        assert out[pos:pos + c] == zref.oracle_compress(src[off:off + n], 1), (off, n)
        pos += c
    assert pos == total


@pytest.mark.parametrize("level", [1, 3])
@pytest.mark.parametrize("size,world", [(5 * (512 << 10) + 12345, 3), (3 << 20, 8), (400_000, 2), (0, 2)])
def test_one_frame_split_over_ranks(ctx, level, size, world):
    """ZSTDB200_compressFramePart: the shares of one frame, each compressed from its own copy of (halo + share) as a rank
    would hold it, concatenate to exactly the frame a single call produces"""
    import torch
    from zstd_b200.sharding import split_one_frame
    L = zstd_b200.lib()
    L.ZSTDB200_framePartHalo.restype = ctypes.c_size_t
    L.ZSTDB200_framePartAlignment.restype = ctypes.c_size_t
    halo, align = L.ZSTDB200_framePartHalo(), L.ZSTDB200_framePartAlignment()
    src = zref.synthetic(size, 17, 0.5)
    whole = ctx.compress(src, level)
    out = b""
    for begin, n in split_one_frame(size, world, align):
        if begin < 0:
            continue
        lo = begin - min(begin, halo)
        part = torch.frombuffer(bytearray(src[lo:begin + n]) or bytearray(1), dtype=torch.uint8).cuda()      # only what the rank holds
        cap = zstd_b200.ZSTD_compressBound(n) + 64
        d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
        k = ctx.compress_frame_part(d_dst.data_ptr(), cap, part.data_ptr(), size, begin, n, level)
        out += bytes(d_dst[:k].cpu().numpy())
    assert out == whole


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary absent")
@pytest.mark.parametrize("level", [2, 4, -1, -7])
def test_size_vs_reference_other_levels(ctx, level):
    """levels the BASELINE configs do not name (2, 4, -1, -7): GPU frame size against the reference's, datagen P30 / P50 / P90, 8 MiB"""
    for p in (30, 50, 90):
        src = zref.datagen(8 << 20, p)
        got = ctx.compress(src, level)
        decode_ok(got, src)
        ref = zref.ref_size(src, level)
        assert zref.size_delta_ok(len(got), ref, len(src)), f"P{p} level {level}: {(len(got) - ref) / ref:+.4%}"


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary absent")
@pytest.mark.parametrize("frame", [4 << 10, 16 << 10, 64 << 10, 256 << 10])
def test_size_vs_reference_small_frames(ctx, frame):
    """frames of 4 KiB .. 256 KiB (32 of each, cut from datagen streams), one batch call per level: summed GPU size against the
    summed reference size (DESIGN.md section 6 lists where this is worst: P90 at 4 KiB, about +6 %)"""
    import torch
    for p in (30, 50, 90):
        big = zref.datagen(16 << 20, p)
        pieces = [big[i * frame:(i + 1) * frame] for i in range(32)]
        src = b"".join(pieces)
        d_src = torch.frombuffer(bytearray(src), dtype=torch.uint8).cuda()
        cap = 32 * (zstd_b200.ZSTD_compressBound(frame) + 32)
        d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
        for level in (1, 3, -3):
            total, csz = ctx.compress_frames(d_dst.data_ptr(), cap, d_src.data_ptr(), [i * frame for i in range(32)], [frame] * 32, level=level)
            ref = sum(zref.ref_size(x, level) for x in pieces)
            assert zref.size_delta_ok(total, ref, frame), f"P{p} frames of {frame} level {level}: {(total - ref) / ref:+.4%}"
