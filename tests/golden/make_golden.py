"""Generates the committed golden fixtures from the compiled reference (run here, where
/root/reference exists):  python tests/golden/make_golden.py
  entropy_vectors.json : (seed, draw) of randomised seqStores -> size + sha256 of the block body the
                         REFERENCE's ZSTD_entropyCompressSeqStore produces
  frames.json          : per input x level: reference compressed size, oracle size + sha256
  inputs/              : the reference's own golden-compression inputs (tests/golden-compression/*) and
                         dictionaries, copied as test data
"""
import json
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import zref  # noqa: E402
from test_oracle_entropy import make_seqstore, run_both  # noqa: E402

REF = "/root/reference/tests"


def main():
    vectors = []
    for seed in (11, 12, 13):
        rng = np.random.default_rng(seed)
        for draw in range(40):
            case = make_seqstore(rng)
            if case is None:
                continue
            r1, h1, r2, b2 = run_both(case)
            assert (r1, h1) == (r2, zref.sha16(b2))
            if 0 < r1 < (1 << 60) and len(vectors) < 40 and draw % 3 == 0:
                vectors.append({"seed": seed, "draw": draw, "size": r1, "sha256": zref.sha(b2)})
    json.dump(vectors, open(os.path.join(HERE, "entropy_vectors.json"), "w"), indent=1)

    os.makedirs(os.path.join(HERE, "inputs"), exist_ok=True)
    for d, names in (("golden-compression", None), ("golden-dictionaries", None), ("dict-files", None)):
        for n in sorted(os.listdir(os.path.join(REF, d))):
            shutil.copyfile(os.path.join(REF, d, n), os.path.join(HERE, "inputs", n))
            os.chmod(os.path.join(HERE, "inputs", n), 0o644)
    frames = {}
    inputs = {n: open(os.path.join(HERE, "inputs", n), "rb").read() for n in
              ("http", "huffman-compressed-larger", "large-literal-and-match-lengths", "PR-3517-block-splitter-corruption-test")}
    inputs["synthetic-300k-seed9"] = zref.synthetic(300000, 9)
    inputs["synthetic-1M-p30-seed4"] = zref.synthetic(1 << 20, 4, 0.3)
    for name, data in inputs.items():
        for level in (1, -1, -3, 3):
            o = zref.oracle_compress(data, level)
            assert zref.ref_decompress(o, len(data)) == data
            frames[f"{name}@{level}"] = {"input_sha256": zref.sha(data), "input_size": len(data),
                                         "ref_size": len(zref.ref_compress(data, level)),
                                         "oracle_size": len(o), "oracle_sha256": zref.sha(o)}
    json.dump(frames, open(os.path.join(HERE, "frames.json"), "w"), indent=1)
    print(len(vectors), "entropy vectors;", len(frames), "frame records")


if __name__ == "__main__":
    main()
