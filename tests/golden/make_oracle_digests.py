#!/usr/bin/env python
"""tests/golden/make_oracle_digests.py — writes tests/golden/oracle_bwt_digests.json: the C oracle's forward transform
(oracle/liboracle.so, the plain-C restatement of BWTManager::doTransform(BWTBlock&, freqs)) of the generated blocks the
GPU tests transform, as SHA-256 digests of the transformed bytes and the freqs, plus the LFpowers, keyed by the digest
of the input and the number of starting points.  A block of up to 256 MiB fits in a few hundred bytes, so the GPU tests
compare full-size blocks with the oracle without running it (a 256 MiB block takes the oracle minutes).
    python tests/golden/make_oracle_digests.py
"""
import json
import os
import sys
from concurrent.futures import ProcessPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

import bwtc_b200 as bw  # noqa: E402
from conftest import Oracle, digest  # noqa: E402

OUT = os.path.join(HERE, "oracle_bwt_digests.json")

# (kind, bytes, seed, starts) of the generated blocks in tests/test_gpu_fullsize.py and tests/test_gpu_inverse.py
GENERATED = ([(k, mib << 20, 31, 8) for k, mib in [("markov", 32), ("dna", 64), ("repetitive", 16), ("random", 256)]]
             + [("random", 64 << 20, 32, 8)]
             + [(k, 32 << 20, 40 + i, 8) for i, k in enumerate(["markov", "dna", "markov", "random"])]
             + [("markov", 32 << 20, 73, 8), ("repetitive", 16 << 20, 73, 8)])


def record(case):
    kind, n, seed, starts = case
    x = bw.generate(kind, n, seed=seed)
    out, LF, fr = Oracle().block(x, starts)
    return "%s:%d" % (digest(x), starts), {"input": "%s n=%d seed=%d" % (kind, n, seed), "bwt": digest(out),
                                           "LF": [int(v) for v in LF], "freqs": digest(fr)}


def main():
    with ProcessPoolExecutor(max_workers=min(len(GENERATED), os.cpu_count() or 1)) as ex:
        rec = dict(ex.map(record, GENERATED))
    with open(OUT, "w") as f:  # one record per line
        f.write("{\n%s\n}\n" % ",\n".join("%s: %s" % (json.dumps(k), json.dumps(rec[k], sort_keys=True)) for k in sorted(rec)))
    print("wrote %d records" % len(rec))


if __name__ == "__main__":
    main()
