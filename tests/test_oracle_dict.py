"""ZSTD_compress_usingDict path of the oracle (BASELINE config 5 shape: small records + shared dictionary).
Frames must decode with the reference's ZSTD_decompress_usingDict and stay within +-0.5 % of the
reference's size for raw-content and zstd-format dictionaries; the dictionary entropy stage (treeless
literals, set_repeat tables, start repcodes) is pinned byte-for-byte against ZSTD_loadCEntropy +
ZSTD_entropyCompressSeqStore of the compiled reference (recorded under tests/golden/reference/ where it is not built)."""
import pytest

import zref

REC = 1024


def records(n, seed, p=0.5):
    data = zref.synthetic(REC * n, seed, p)
    return [data[i * REC:(i + 1) * REC] for i in range(n)]


@pytest.mark.parametrize("dict_name", ["zdict-16k-synthetic-seed77", "http-dict-missing-symbols", "zero-weight-dict"])
def test_zstd_format_dictionaries_roundtrip(dict_name):
    d = zref.golden_input(dict_name)
    tot_o = tot_r = 0
    srcs = records(200, 5) + [b"", b"a", zref.golden_input("http"), zref.synthetic(300_000, 8)]
    for src in srcs:
        f = zref.oracle_compress_using_dict(src, d, 1)
        assert zref.ref_decodes(f, src, d)
        assert f[4] & 3, "dictID must be present in the frame header for a zstd-format dictionary"
        tot_o += len(f)
        tot_r += zref.ref_size(src, 1, d)
    if dict_name.startswith('zdict'):
        assert abs(tot_o - tot_r) / tot_r <= 0.01, (tot_o, tot_r)
    else:
        assert tot_o < tot_r * 1.03          # tiny hand-made dictionaries of the reference's test suite


def test_raw_content_dictionary_size_parity():
    d = zref.synthetic(32 << 10, 123, 0.5)                 # no magic number -> raw content (zstd_compress.c:5143-5148)
    tot_o = tot_r = 0
    for src in records(400, 6):
        f = zref.oracle_compress_using_dict(src, d, 1)
        assert zref.ref_decodes(f, src, d)
        assert (f[4] & 3) == 0                              # no dictID for raw content (lib/zstd.h:185-186)
        tot_o += len(f)
        tot_r += zref.ref_size(src, 1, d)
    assert abs(tot_o - tot_r) / tot_r <= 0.01


def test_dictionary_content_is_actually_used():
    """A record that is a verbatim slice of the dictionary must compress to almost nothing."""
    d = zref.synthetic(32 << 10, 321, 0.1)
    src = d[5000:6024]
    with_dict = zref.oracle_compress_using_dict(src, d, 1)
    without = zref.oracle_compress(src, 1)
    assert zref.ref_decodes(with_dict, src, d)
    assert len(with_dict) < 100 < len(without)


def test_short_and_corrupted_dictionaries():
    src = zref.synthetic(5000, 1)
    assert zref.oracle_compress_using_dict(src, b"1234567", 1) == zref.oracle_compress(src, 1)      # < 8 bytes: ignored
    bad = bytes.fromhex("37a430ec01000000") + bytes(40)
    with pytest.raises(RuntimeError, match="30"):                                                     # dictionary_corrupted
        zref.oracle_compress_using_dict(src, bad, 1)


@pytest.mark.parametrize("dict_name", ["zdict-16k-synthetic-seed77", "http-dict-missing-symbols", "zero-weight-dict"])
def test_dictionary_entropy_stage_byte_exact(dict_name):
    """oracle/zb_dict.c + zbo_entropyCompressBlock_prev vs the reference's ZSTD_loadCEntropy (zstd_compress.c:4987)
    + ZSTD_entropyCompressSeqStore (:3001) on randomised seqStores, through oracle/ref_shim.c."""
    import ctypes
    import numpy as np
    from test_oracle_entropy import make_seqstore
    O = zref.oracle()
    c_sz, vp = ctypes.c_size_t, ctypes.c_void_p
    O.zbo_loadDictEntropy.restype = c_sz
    O.zbo_loadDictEntropy.argtypes = [vp, vp, c_sz]
    O.zbo_entropyCompressBlock_prev.restype = c_sz
    O.zbo_entropyCompressBlock_prev.argtypes = [vp, c_sz, vp, c_sz, vp, c_sz, c_sz, ctypes.c_uint, ctypes.c_int, vp]
    d = zref.golden_input(dict_name)
    de = ctypes.create_string_buffer(16384)
    assert 8 < O.zbo_loadDictEntropy(de, d, len(d)) < len(d)
    rng = np.random.default_rng(5)
    compressed = 0
    for t in range(250):
        case = make_seqstore(rng)
        if case is None:
            continue
        offb, ll, ml, lits, block, strategy, tl = case
        if t % 2 == 0:                                             # the small-record regime (preferRepeat, set_repeat)
            k = max(1, min(len(offb), 40))
            offb, ll, ml = offb[:k], ll[:k], ml[:k]
            lits = lits[:min(len(lits), int(ll.sum()) + 50)]
            if int(ll.sum()) > len(lits):
                continue
            block = max(7, min(131072, len(lits) + int(ml.sum())))
        nseq = len(offb)
        cap = 1 << 20
        d1, d2 = ctypes.create_string_buffer(cap), ctypes.create_string_buffer(cap)
        seqs = np.ascontiguousarray(np.stack([offb, ll, ml], axis=1).astype(np.uint32)) if nseq else np.zeros((0, 3), np.uint32)
        offb, ll, ml = (np.ascontiguousarray(a, dtype=np.uint32) for a in (offb, ll, ml))
        lits = np.ascontiguousarray(lits)
        tlv = tl if strategy == 1 else 0
        def reference():
            R = zref.ref()
            R.ref_entropyCompressBlock_dict.restype = c_sz
            R.ref_entropyCompressBlock_dict.argtypes = [vp, c_sz, vp, vp, vp, c_sz, vp, c_sz, c_sz, ctypes.c_int, ctypes.c_uint, vp, c_sz]
            r = R.ref_entropyCompressBlock_dict(d1, cap, offb.ctypes.data, ll.ctypes.data, ml.ctypes.data, nseq, lits.ctypes.data, len(lits), block, 1, tlv, d, len(d))
            return [r, zref.sha16(d1.raw[:r]) if r < (1 << 60) else None]
        r1, h1 = zref.recorded(zref._key("entropy-dict", seqs.tobytes(), lits.tobytes(), block, tlv, d), reference)
        with zref.entropy_model(0):                                 # the restatement of the reference's table builders
            r2 = O.zbo_entropyCompressBlock_prev(d2, cap, seqs.ctypes.data, nseq, lits.ctypes.data, len(lits), block, 1, 1 if tlv > 0 else 0, de)
        assert r1 == r2
        if r1 < (1 << 60):
            assert h1 == zref.sha16(d2.raw[:r2])
            compressed += r1 > 0
    assert compressed > 80


@pytest.mark.skipif(not zref.have_datagen(), reason="oracle/_ref/datagen not built")
@pytest.mark.parametrize("level", [1, 3, -3])
def test_size_parity_with_reference_cdict(level):
    """ZSTD_compress_usingCDict is the production form of config 5 (SURVEY.md §8f rank 1).  The GPU CDict path
    emits the bytes of the usingDict path, so the oracle's usingDict output must sit within +-1 % of what the
    reference's ZSTD_compress_usingCDict produces on config 5's data (datagen -P50 cut into 1 KiB records,
    16 KiB ZDICT dictionary) — including level 3, where both run doubleFast over a dictionary."""
    data = zref.datagen(REC * 6000, 50)
    d = zref.train_dict(data, REC, 4000, 16 << 10)
    srcs = [data[i * REC:(i + 1) * REC] for i in range(4000, 5000)]
    tot_o = 0
    for k, src in enumerate(srcs):
        f = zref.oracle_compress_using_dict(src, d, level)
        if k % 25 == 0:
            assert zref.ref_decodes(f, src, d)
        tot_o += len(f)
    tot_r = zref.ref_cdict_size(srcs, d, level)
    assert abs(tot_o - tot_r) / tot_r <= 0.01, (tot_o, tot_r)
