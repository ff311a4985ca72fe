"""GPU parity at BASELINE.json's block sizes: the CUDA path (C-ABI, block contract) against the C oracle's outputs
(oracle/oracle_bwt.c, the restatement of BWTManager('d'), itself pinned to the unmodified reference by
tests/test_oracle.py), recorded in tests/golden/oracle_bwt_digests.json — bit-exact (bytes, LFpowers, freqs), not
properties.
The paths that only switch on by size run here: the one-byte predecessor payload (>= 96 M suffixes), the bucketed rank
scatter (>= 3 L2 windows), 7/8-pass doubling keys, global radix rounds over tens of millions of records.
Also real (non-synthetic) source text, and a short randomized soak of pipeline vs single context."""
import numpy as np
import pytest

import bwtc_b200 as bw
from _inputs import real_source_text

pytestmark = pytest.mark.gpu


def _gpu_block(x, starts=8):
    n = x.size
    ctx = bw.CudaContext(n)
    try:
        blk = np.concatenate([x, np.array([0x5A], np.uint8)])
        view = blk[:-1]
        LF = np.zeros(bw.num_starting_points(n, starts), np.uint32)
        fr = np.zeros(256, np.uint32)
        pidx = ctx.bwt_block(view, LF, fr)
        st = ctx.stats()
    finally:
        ctx.close()
    assert blk[-1] == 0x5A, "byte after the block must be preserved"
    assert pidx == LF[0]
    return view, LF, fr, st


def _compare_with_record(oracle_record, x, starts=8):
    view, LF, fr, st = _gpu_block(x, starts)
    oracle_record.check(x, starts, view, LF, fr)
    return st


@pytest.mark.parametrize("kind,mib", [("markov", 32), ("dna", 64), ("repetitive", 16), ("random", 256)])
def test_baseline_block_sizes_bit_exact_vs_reference(oracle_record, kind, mib):
    """BASELINE.json configs 5/bench, 2, 3, 4: one full-size block each, compared byte for byte."""
    x = bw.generate(kind, mib << 20, seed=31)
    st = _compare_with_record(oracle_record, x)
    assert st["n_suffixes"] == (mib << 20) + 1 and st["live"][0] == st["n_suffixes"]
    if kind == "random":
        assert st["flags"] & 8, "256 MiB of bytes: the predecessor codes should travel as a one-byte payload"
    if kind == "repetitive":
        assert max(st["passes"][1:]) >= 5, "the repetitive block should need global radix rounds"


def test_random_64mib_bit_exact_vs_reference(oracle_record):
    """64 MiB of random bytes: no spare id bits, text gather at emission, bucketed scatter with 4 windows."""
    _compare_with_record(oracle_record, bw.generate("random", 64 << 20, seed=32))


def test_real_source_text_32mib_bit_exact_vs_reference(oracle):
    """Non-synthetic, LCP-heavy data (14-15 rounds, 6-8 of them global radix rounds).  The text is whatever this Python
    installation holds, so nothing is recorded for it: the C oracle transforms it here."""
    x = real_source_text(32 << 20)
    if x.size < (8 << 20):
        pytest.skip("not enough source text in this image")
    view, LF, fr, st = _gpu_block(x)
    want_bytes, want_LF, want_fr = oracle.block(x, 8)
    assert (LF == want_LF).all(), (LF, want_LF)
    assert (fr == want_fr).all()
    assert np.array_equal(view, want_bytes), "BWT bytes differ from the oracle's"
    assert st["rounds"] >= 4


def test_pipeline_full_size_blocks_equal_reference(oracle_record):
    """The batched look-ahead path (bwtc_cuda_pipeline_run, several blocks in flight) at 32 MiB: every block equals the
    oracle's recorded output — the pipeline never reorders or mixes results."""
    n = 32 << 20
    blocks = [bw.generate(k, n, seed=40 + i) for i, k in enumerate(["markov", "dna", "markov", "random"])]
    pipe = bw.Pipeline(n, depth=3)
    try:
        work = [b.copy() for b in blocks]
        LF, nLF, freqs, stats = pipe.run(work, starts=8)
    finally:
        pipe.close()
    for i, x in enumerate(blocks):
        oracle_record.check(x, 8, work[i], LF[i, : nLF[i]], freqs[i])


def test_soak_pipeline_equals_single_context():
    """Randomized mixes of kinds / sizes / depths through the pipeline (batches of small blocks included) and one by one
    through a single context: identical bytes, LFpowers, freqs (a short version of tests/gpu_soak.py)."""
    rng = np.random.default_rng(2)
    kinds = ["markov", "dna", "repetitive", "random"]
    cap = 4 << 20
    single = bw.CudaContext(cap)
    pipes = {}
    flags_seen = 0
    try:
        for it in range(10):
            nb = int(rng.integers(4, 24))
            if it % 2 == 0:  # a run of equal-sized small blocks (gets batched), last one shorter
                n0 = int(rng.integers(1, 1 << 18))
                sizes = [n0] * (nb - 1) + [int(rng.integers(1, n0 + 1))]
            else:
                sizes = [int(2 ** rng.uniform(0, 22)) for _ in range(nb)]
            kind = kinds[it % 4]
            blocks = [bw.generate(kind, max(1, s), seed=int(rng.integers(0, 1 << 30))) for s in sizes]
            if it % 3 == 0:
                for b in blocks:
                    b[rng.integers(0, b.size, max(1, b.size // 50))] = 0
            depth = 1 + it % 4
            if depth not in pipes:
                pipes[depth] = bw.Pipeline(cap, depth=depth)
            work = [b.copy() for b in blocks]
            LF, nLF, fr, stats = pipes[depth].run(work, 8)
            for i, b in enumerate(blocks):
                w = b.copy()
                k = bw.num_starting_points(b.size, 8)
                lf1 = np.zeros(k, np.uint32)
                fr1 = np.zeros(256, np.uint32)
                single.bwt_block(w, lf1, fr1)
                flags_seen |= single.stats()["flags"] | stats[i]["flags"]
                assert (w == work[i]).all() and nLF[i] == k and (LF[i, :k] == lf1).all() and (fr[i] == fr1).all(), (it, kind, i)
    finally:
        single.close()
        for p in pipes.values():
            p.close()
    assert not (flags_seen & 1), "unexpected look-back watchdog fallback during the soak"
