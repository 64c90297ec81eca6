"""Oracle at frame level: every frame decodes with the reference decoder, sizes stay within the
two-sided bound of zref.size_delta_ok on the BASELINE inputs, parameter derivation equals the reference's, golden fixtures.
The reference's answers come from the compiled library where it is built and from tests/golden/reference/ elsewhere."""
import ctypes
import json
import os

import pytest

import zref

@pytest.mark.parametrize("level", [1, 2, 3, 4, 0, -1, -3, -7])
@pytest.mark.parametrize("size", [0, 1, 100, 1000, 16 << 10, (16 << 10) + 1, 100_000, 128 << 10, (128 << 10) + 1,
                                  256 << 10, (256 << 10) + 1, 1 << 20, 5 << 20, 600 << 20])
def test_cparams_match_reference(level, size):
    """zbo_getCParams restates ZSTD_getCParams_internal + ZSTD_adjustCParams_internal
    (zstd_compress.c:7123-7146, :1465-1602) for rows whose strategy is fast/dfast."""
    class CP(ctypes.Structure):
        _fields_ = [(n, ctypes.c_uint) for n in ("windowLog", "chainLog", "hashLog", "searchLog", "minMatch", "targetLength", "strategy")]
    O = zref.oracle()
    O.zbo_getCParams.restype = CP
    O.zbo_getCParams.argtypes = [ctypes.c_int, ctypes.c_ulonglong, ctypes.c_size_t]
    def reference():
        out = (ctypes.c_uint * 7)()
        zref.ref().ref_getCParams_simpleApi(level, size, 0, out)
        return list(out)
    out = zref.recorded(zref._key("cparams", level, size), reference)
    ours = O.zbo_getCParams(level, size, 0)
    if out[6] > 2:
        pytest.skip("reference strategy above dfast: out of scope, served by the dfast row")
    assert [ours.windowLog, ours.chainLog, ours.hashLog, ours.searchLog, ours.minMatch, ours.targetLength, ours.strategy] == out


def test_compress_bound_matches_reference():
    O = zref.oracle()
    for n in [0, 1, 100, 1 << 10, 128 << 10, (128 << 10) - 1, (128 << 10) + 1, 1 << 20, 1 << 30, 5 << 30]:
        assert O.zbo_compressBound(n) == zref.ref_call("ZSTD_compressBound", n)


EDGE = {
    "empty": b"", "one": b"x", "six": b"abcdef", "seven": b"abcdefg",
    "zeros-300": bytes(300), "zeros-1M": bytes(1 << 20), "zeros-128k+1": bytes((128 << 10) + 1),
    "rand-100k": zref.random_bytes(100_000, 1), "rand-300k": zref.random_bytes(300_000, 2),
    "period3": b"abc" * 50_000, "syn-128k": zref.synthetic(128 << 10, 3), "syn-128k+1": zref.synthetic((128 << 10) + 1, 3),
    "syn-1M-p90": zref.synthetic(1 << 20, 5, 0.9), "syn-1M-p10": zref.synthetic(1 << 20, 6, 0.1),
}
# sizes around the 16 KiB parse-segment boundaries (a segment end within 8 bytes of the block end, one byte past it, ...)
SEG = 16 << 10
for _n in (SEG - 1, SEG, SEG + 1, SEG + 6, SEG + 7, SEG + 8, 2 * SEG + 3, 8 * SEG - 1, 8 * SEG + SEG + 5, 3 * 8 * SEG + 9):
    EDGE[f"seg-{_n}"] = zref.synthetic(_n, 40 + _n % 7, 0.6)
EDGE["seg-rep"] = (zref.synthetic(5000, 77, 0.3) * 30)[: 9 * SEG + 123]        # matches that want to run across every segment end


@pytest.mark.parametrize("name", sorted(EDGE))
@pytest.mark.parametrize("level", [1, -3, 3])
def test_roundtrip_edge_cases(name, level):
    src = EDGE[name]
    frame = zref.oracle_compress(src, level)
    assert zref.ref_decodes(frame, src)
    assert len(frame) <= zref.ref_call("ZSTD_compressBound", len(src))
    assert zref.ref_frame_content_size(frame) == len(src)                           # fuzzer.c:4565-4573
    assert zref.oracle_compress(src, level) == frame                                  # determinism (fuzz/simple_round_trip.c)


def test_dst_too_small_is_an_error_not_an_overflow():
    src = zref.synthetic(300_000, 1)
    full = zref.oracle_compress(src, 1)
    O = zref.oracle()
    for cap in (0, 5, 17, 18, 100, len(full) - 1):
        dst = ctypes.create_string_buffer(cap + 64)
        ctypes.memset(dst, 0xA5, cap + 64)
        r = O.zbo_compress(dst, cap, src, len(src), 1)
        assert r == (1 << 64) - 70, f"cap={cap}: expected dstSize_tooSmall"
        assert dst.raw[cap:] == b"\xa5" * 64                                         # fuzzer.c:4550-4562
    dst = ctypes.create_string_buffer(len(full))
    assert O.zbo_compress(dst, len(full), src, len(src), 1) == len(full)


def test_golden_frames_fixture():
    """tests/golden/frames.json (from tests/golden/make_golden.py): the oracle reproduces its recorded
    output on the reference's golden-compression inputs; recorded reference sizes document the gap."""
    frames = json.load(open(os.path.join(zref.GOLDEN, "frames.json")))
    for key, rec in frames.items():
        name, level = key.rsplit("@", 1)
        path = os.path.join(zref.GOLDEN, "inputs", name)
        if os.path.exists(path):
            data = open(path, "rb").read()
        elif name == "synthetic-300k-seed9":
            data = zref.synthetic(300000, 9)
        elif name == "synthetic-1M-p30-seed4":
            data = zref.synthetic(1 << 20, 4, 0.3)
        else:
            raise AssertionError(name)
        assert zref.sha(data) == rec["input_sha256"]
        out = zref.oracle_compress(data, int(level))
        assert len(out) == rec["oracle_size"] and zref.sha(out) == rec["oracle_sha256"], key
        assert zref.size_delta_ok(len(out), rec["ref_size"], len(data), name.startswith("synthetic")), (key, len(out), rec["ref_size"])
        assert zref.ref_decodes(out, data)
        assert zref.ref_size(data, int(level)) == rec["ref_size"]


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary not built")
@pytest.mark.parametrize("p,level,size", [(50, 1, 16 << 20), (30, -3, 16 << 20), (90, 3, 64 << 20)])
def test_size_close_to_reference(p, level, size):
    """BASELINE.json configs 1/2 (P50, level 1), 3 (P30, --fast=3) and 4 (P90, level 3) on 16 / 64 MiB samples:
    inside the two-sided bound of zref.size_delta_ok (measured: -0.65 %, -0.3 %, -1.2 %)."""
    src = zref.datagen(size, p)
    ours = zref.oracle_compress(src, level)
    ref = zref.ref_size(src, level)
    assert zref.ref_decodes(ours, src)
    delta = (len(ours) - ref) / ref
    assert zref.size_delta_ok(len(ours), ref, len(src)), f"size delta {delta:+.4%} (ours {len(ours)}, reference {ref})"


@pytest.mark.skipif(not zref.have_datagen(), reason="reference datagen binary not built")
@pytest.mark.parametrize("level", [1, 3, -3])
@pytest.mark.parametrize("p", [30, 50, 90])
def test_one_rule_for_all_datagen_types(p, level):
    """the same table sizes and insertion rule serve P30, P50 and P90 (round 1 fitted level 3 to P90 alone): 8 MiB samples"""
    src = zref.datagen(8 << 20, p)
    ours = zref.oracle_compress(src, level)
    ref = zref.ref_size(src, level)
    assert zref.ref_decodes(ours, src)
    assert zref.size_delta_ok(len(ours), ref, len(src)), f"{(len(ours) - ref) / ref:+.4%}"
