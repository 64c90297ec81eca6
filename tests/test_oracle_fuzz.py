"""Seeded differential fuzz of the oracle against the reference decoder (CPU): structured random inputs whose sizes
cluster around the 16 KiB parse-segment and 128 KiB block boundaries, all level classes, with and without a zstd-format
dictionary.  The reference decoder's verdicts are recorded under tests/golden/reference/ for machines without it.  A longer run of the same generator (400 k cases) and its GPU twin (tests/fuzz_gpu.py) are recorded in
profiles/r1_sanitizer.txt."""
import random

import pytest

import zref

def make_input(rng):
    kind = rng.randrange(6)
    size = rng.choice([rng.randrange(0, 300), rng.randrange(0, 40000), rng.randrange(16000, 17000), rng.randrange(130000, 133000),
                       rng.randrange(0, 400000)])
    if kind == 0:
        return zref.synthetic(size, rng.randrange(1 << 30), rng.random())
    if kind == 1:
        return zref.random_bytes(size, rng.randrange(1 << 30))
    if kind == 2:
        return bytes([rng.randrange(256)]) * size
    if kind == 3:
        unit = zref.random_bytes(rng.randrange(1, 5000), rng.randrange(1 << 30))
        return (unit * (size // max(1, len(unit)) + 1))[:size]
    if kind == 4:
        a = zref.synthetic(size // 2 + 1, rng.randrange(1 << 30), 0.95)
        return (a + zref.random_bytes(size // 2 + 1, rng.randrange(1 << 30)) + a)[:size]
    return zref.synthetic(size, rng.randrange(1 << 30), 0.99)


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_oracle_frames_decode(seed):
    rng = random.Random(seed)
    d = zref.golden_input("zdict-16k-synthetic-seed77")
    for _ in range(400):
        src = make_input(rng)
        level = rng.choice([1, 2, 3, 4, -1, -3, -7, -50, 0, 9])
        if rng.random() < 0.25:
            frame = zref.oracle_compress_using_dict(src, d, level)
            assert zref.ref_decodes(frame, src, d), (len(src), level)
        else:
            frame = zref.oracle_compress(src, level)
            assert zref.ref_decodes(frame, src), (len(src), level)
