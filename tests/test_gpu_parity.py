"""GPU parity tests (the first gate): the CUDA path, called through the C-ABI, must be bit-exact with the oracle
on the same seeded inputs and with the golden fixtures generated from the reference.  BASELINE.json's block sizes
are compared bit for bit with the compiled reference in tests/test_gpu_fullsize.py; the engine's maximum block size
(no CPU checker finishes in test time) is covered by size-independent properties here."""
import numpy as np
import pytest

import bwtc_b200 as bw

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(4 << 20)
    yield c
    c.close()


def _gpu_block(ctx, x, starts, want_freqs=True):
    blk = np.concatenate([x, np.array([0xAB], np.uint8)])
    view = blk[:-1]
    LF = np.zeros(bw.num_starting_points(x.size, starts), np.uint32)
    fr = np.zeros(256, np.uint32) if want_freqs else None
    pidx = ctx.bwt_block(view, LF, fr)
    assert blk[-1] == 0xAB, "byte after the block must be preserved"
    assert pidx == LF[0]
    return view.copy(), LF, fr


def test_golden_fixtures(ctx, golden):
    for name, g in golden.items():
        out, LF, fr = _gpu_block(ctx, g["in"], int(g["starts"][0]))
        assert (out == g["out"]).all(), name
        assert (LF == g["LF"]).all(), name
        assert (fr == g["freqs"]).all(), name


def test_block_contract_vs_oracle_random(ctx, oracle):
    rng = np.random.default_rng(11)
    sizes = [1, 2, 3, 4, 7, 8, 9, 31, 32, 33, 255, 256, 257, 258, 1000, 2047, 2048, 2049, 4095, 4096, 4097, 8191, 8192,
             8193, 10000, 65535, 65536, 65537, 200000]
    for n in sizes:
        for sigma in (1, 2, 3, 4, 5, 64, 255, 256):
            x = rng.integers(0, sigma, n).astype(np.uint8)
            if sigma == 5:
                x += 1  # no 0x00 in the block: the sentinel stays outside the alphabet
            starts = int(rng.choice([1, 2, 7, 8, 256]))
            want = oracle.block(x, starts)
            got = _gpu_block(ctx, x, starts)
            assert (got[0] == want[0]).all(), (n, sigma, starts)
            assert (got[1] == want[1]).all(), (n, sigma, starts)
            assert (got[2] == want[2]).all(), (n, sigma, starts)


def test_freqs_are_incremented_not_overwritten(ctx):
    x = np.frombuffer(b"abracadabra", np.uint8).copy()
    LF = np.zeros(1, np.uint32)
    fr = np.full(256, 5, np.uint32)
    ctx.bwt_block(x.copy(), LF, fr)
    assert fr[ord("a")] == 10 and fr[ord("z")] == 5


def test_structured_inputs_vs_oracle(ctx, oracle):
    rng = np.random.default_rng(12)
    cases = {
        "all zero": np.zeros(5000, np.uint8),
        "all equal": np.full(70000, 0x41, np.uint8),
        "ab*k": np.frombuffer(b"ab" * 30000, np.uint8).copy(),
        "abc*k+z": np.frombuffer(b"abc" * 20000 + b"z", np.uint8).copy(),
        "many zeros": np.where(rng.random(50000) < 0.9, 0, rng.integers(0, 256, 50000)).astype(np.uint8),
        "zero tail": np.concatenate([rng.integers(1, 256, 3000), np.zeros(3000)]).astype(np.uint8),
        "zero head": np.concatenate([np.zeros(3000), rng.integers(1, 256, 3000)]).astype(np.uint8),
        "fibonacci": None,
        "tiled+mut": None,
        "descending": (255 - (np.arange(100000) % 256)).astype(np.uint8),
    }
    a, b = b"a", b"ab"
    while len(b) < 100000:
        a, b = b, b + a
    cases["fibonacci"] = np.frombuffer(b[:100000], np.uint8).copy()
    t = np.tile(rng.integers(0, 256, 777).astype(np.uint8), 200)
    t[rng.integers(0, t.size, 100)] = 7
    cases["tiled+mut"] = t
    for name, x in cases.items():
        for starts in (1, 8):
            want = oracle.block(x, starts)
            got = _gpu_block(ctx, x, starts)
            assert (got[0] == want[0]).all() and (got[1] == want[1]).all() and (got[2] == want[2]).all(), (name, starts)


@pytest.mark.parametrize("kind", ["markov", "dna", "repetitive", "random"])
def test_input_families_1mib_vs_oracle(ctx, oracle, kind):
    x = bw.generate(kind, 1 << 20, seed=21)
    want = oracle.block(x, 8)
    got = _gpu_block(ctx, x, 8)
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all() and (got[2] == want[2]).all()


@pytest.mark.parametrize("force", [(0, 0), (1, 4), (3, 4), (2, 8), (5, 8), (64, 8)])
def test_any_round0_key_shape_gives_identical_bytes(ctx, oracle, force):
    """The round-0 key shape is a performance knob only."""
    x = bw.generate("markov", 150001, seed=22)
    want = oracle.block(x, 8)
    ctx.set_round0(*force)
    try:
        got = _gpu_block(ctx, x, 8)
    finally:
        ctx.set_round0(0, 0)
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all()


@pytest.mark.parametrize("gram", ["1", "0"])
@pytest.mark.parametrize("sigma,force", [(8, (0, 0)), (8, (4, 4)), (7, (5, 4)), (8, (10, 4)), (5, (12, 8)), (8, (21, 8)),
                                         (64, (2, 4)), (64, (3, 4)), (33, (7, 8)), (64, (10, 8))])
def test_round0_histograms_from_the_gram_histogram(oracle, monkeypatch, gram, sigma, force):
    """3-bit and 6-bit codes: k_pack_round0 counts ONE 4096-bin histogram of the keys' last 4 / 2 characters and every digit
    histogram of the round-0 sort is projected from it (BWTC_GRAM=0: per-digit counting + k_hist_derive).  A wrong
    histogram sends records to wrong places, so the bytes are the check; sizes with ragged tiles, text ending in the smallest
    and in the largest symbol (the zero padding past the end is part of the windows that are counted)."""
    monkeypatch.setenv("BWTC_GRAM", gram)
    if sigma % 2:  # odd alphabet sizes also run without the partial character in the spare key bits
        monkeypatch.setenv("BWTC_PARTIAL", "0")
    rng = np.random.default_rng(1000 + sigma)
    for n, tail in ((70001, 0), (300007, sigma - 1), (65, 1)):
        x = rng.integers(0, sigma, n).astype(np.uint8)
        x[-30:] = tail
        x[: sigma] = np.arange(sigma, dtype=np.uint8)  # every symbol present: the code width is what the case says
        want = oracle.block(x, 8)
        c = bw.CudaContext(n + 1)
        c.set_round0(*force)
        try:
            got = _gpu_block(c, x, 8)
        finally:
            c.close()
        assert (got[0] == want[0]).all() and (got[1] == want[1]).all() and (got[2] == want[2]).all(), (n, tail)


@pytest.mark.parametrize("radix9", ["1", "0"])
@pytest.mark.parametrize("kind,chars", [("markov", 6), ("markov", 7), ("markov", 8), ("markov", 9), ("markov", 10),
                                        ("dna", 17), ("dna", 22), ("dna", 27), ("dna", 31), ("dna", 32),
                                        ("random", 5), ("random", 8)])
def test_digit_width_of_the_radix_passes(oracle, monkeypatch, radix9, kind, chars):
    """64-bit keys of 34..64 used bits: with BWTC_RADIX9=1 (an experiment, measured slower, default off) 9-bit digits are
    chosen whenever they save a pass over 8-bit digits (36 bits: 4 instead of 5 passes, ... 60 bits: 7 instead of 8; 48 and
    64 bits: 8-bit digits stay).  Same bytes either way, and
    the pass count of round 0 shows which width ran.  A size with a ragged last tile and >= 2 tiles per CTA wave."""
    monkeypatch.setenv("BWTC_RADIX9", radix9)
    n = 700001
    x = bw.generate(kind, n, seed=29)
    want = oracle.block(x, 8)
    c = bw.CudaContext(n + 1)
    c.set_round0(chars, 8)
    try:
        got = _gpu_block(c, x, 8)
        st = c.stats()
    finally:
        c.close()
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all() and (got[2] == want[2]).all()
    bits = {"markov": 6, "dna": 2, "random": 8}[kind] * chars
    p8, p9 = -(-bits // 8), -(-bits // 9)
    assert st["passes"][0] == (p9 if (radix9 == "1" and p9 < p8) else p8), (bits, st["passes"][:2])


@pytest.mark.parametrize("force", [(0, 0), (1, 4), (3, 4), (2, 8), (5, 8), (64, 8)])
@pytest.mark.parametrize("kind", ["markov", "dna", "zeros"])
def test_lazy_ranks_with_any_key_shape(oracle, monkeypatch, force, kind):
    """Lazy ranks forced (BWTC_LAZY=2) under every round-0 key shape: short keys leave nearly every suffix in a group
    (more than the lazy list pool holds -> fallback, ranks materialised), long keys leave few (looked up in the sorted
    keys); text ending in / consisting of zeros exercises the 'short suffix' rule.  Always the oracle's bytes."""
    monkeypatch.setenv("BWTC_LAZY", "2")
    if kind == "zeros":
        x = np.zeros(100003, np.uint8)
        x[::977] = 1
    else:
        x = bw.generate(kind, 300007, seed=23)
        x[-40:] = x[0]
    want = oracle.block(x, 8)
    c = bw.CudaContext(x.size + 1)
    c.set_round0(*force)
    try:
        got = _gpu_block(c, x, 8)
        raw = np.concatenate([x[::-1], np.zeros(1, np.uint8)])  # the raw contract goes through the same machinery
        LFr = np.zeros(8, np.uint32)
        frr = np.zeros(256, np.uint32)
        rc, wbuf, wLF, wfr = oracle.raw(raw, 8)
        U = raw.copy()
        assert c.divbwtf(U, U, LFr, frr) == rc and (U == wbuf).all() and (LFr == wLF).all()
    finally:
        c.close()
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all() and (got[2] == want[2]).all()


def test_raw_contract_vs_oracle(ctx, oracle):
    """doTransform(byte* begin, uint32 length, vector<uint32>& LF, freqs) on a caller-prepared buffer, as
    test/InverseBwtTest.cpp:57-66 calls it; arbitrary last byte allowed (same semantics as divbwtf)."""
    rng = np.random.default_rng(13)
    for trial in range(60):
        n = int(rng.integers(2, 20000))
        sigma = int(rng.choice([1, 2, 4, 16, 256]))
        T = rng.integers(0, sigma, n).astype(np.uint8)
        if trial % 2 == 0:
            T[-1] = 0  # the reference's own usage: reverse(text) + '\0'
        nLF = int(rng.integers(1, min(n, 256) + 1))
        rc, wbuf, wLF, wfr = oracle.raw(T, nLF)
        U = T.copy()
        LF = np.zeros(nLF, np.uint32)
        fr = np.zeros(256, np.uint32)
        pidx = ctx.divbwtf(U, U, LF, fr)
        assert pidx == rc and (U == wbuf).all() and (LF == wLF).all() and (fr == wfr).all(), (trial, n, sigma, nLF)
    # n <= 1 early-out (divsufsort.c:488-489): LFpowers untouched, returns n
    U = np.array([9], np.uint8)
    LF = np.array([77], np.uint32)
    assert ctx.divbwtf(U, U, LF, None) == 1 and LF[0] == 77 and U[0] == 9


def test_error_behaviour(ctx):
    small = bw.CudaContext(1000)
    with pytest.raises(bw.BwtcCudaError) as e:
        small.bwt_block(np.zeros(2000, np.uint8), np.zeros(8, np.uint32), None)
    assert e.value.code == -5
    with pytest.raises(bw.BwtcCudaError) as e:  # nLF > N: x = N / nLF would be 0 (UB in the reference)
        small.divbwtf(np.zeros(4, np.uint8), np.zeros(4, np.uint8), np.zeros(8, np.uint32), None)
    assert e.value.code == -1
    small.close()


def test_manager_interface_matches_oracle(oracle):
    """Reads like the reference's own use: BWTManager m(starts); m.initialize(c); m.doTransform(block, freqs)."""
    x = bw.generate("markov", 300000, seed=23)
    want = oracle.block(x, 8)
    m = bw.BWTManager(8, max_block_bytes=x.size)
    m.initialize("c")
    data = x.copy()
    block = bw.BWTBlock(data)
    fr = np.zeros(256, np.uint32)
    m.doTransform(block, fr)
    assert block.isTransformed()
    assert (data == want[0]).all() and (block.LFpowers() == want[1]).all() and (fr == want[2]).all()


def test_pipeline_equals_single_context(oracle):
    rng = np.random.default_rng(14)
    sizes = [1, 300, 70000, 1 << 18, 123457, 1 << 18, 999, 1 << 17]
    blocks = [bw.generate(["markov", "dna", "repetitive", "random"][i % 4], s, seed=100 + i) for i, s in enumerate(sizes)]
    want = [oracle.block(b, 8) for b in blocks]
    pipe = bw.Pipeline(1 << 18, depth=3)
    work = [b.copy() for b in blocks]
    LF, nLF, freqs, stats = pipe.run(work, starts=8)
    for i, w in enumerate(want):
        assert (work[i] == w[0]).all(), i
        assert (LF[i, : nLF[i]] == w[1]).all(), i
        assert (freqs[i] == w[2]).all(), i
        assert stats[i]["n_suffixes"] >= sizes[i] + 1  # (== for a block on its own, the batch's total when batched)
    pipe.close()


def _check_batch(ctx, oracle, blocks, starts):
    want = [oracle.block(x, starts) for x in blocks]
    work = [x.copy() for x in blocks]
    LF, nLF, fr = ctx.bwt_blocks(work, starts)
    for k, w in enumerate(want):
        assert (work[k] == w[0]).all(), ("bwt", k)
        assert nLF[k] == w[1].size and (LF[k, : nLF[k]] == w[1]).all(), ("LF", k)
        assert (fr[k] == w[2]).all(), ("freqs", k)
    return ctx.stats()


def test_batched_small_blocks_equal_single_blocks(oracle):
    """bwtc_cuda_bwt_blocks sorts runs of equal-sized blocks as ONE text (block number above the key, reserved
    sentinel code): every block's (bytes, LFpowers, freqs) must equal what the block gets on its own."""
    rng = np.random.default_rng(5)
    ctx = bw.CudaContext(8 << 20)
    try:
        # 16 x 256 KiB Markov blocks, last one shorter: one batch
        blocks = [bw.generate("markov", 1 << 18, seed=100 + k) for k in range(15)] + [bw.generate("markov", 77777, seed=99)]
        st = _check_batch(ctx, oracle, blocks, 8)
        assert st["n_suffixes"] == 15 * ((1 << 18) + 1) + 77778, "the run must have been transformed as one batch"
        # data full of 0x00 (the sentinel's byte value), two-letter and one-letter blocks, repeats across blocks
        z = [rng.integers(0, 3, 50000).astype(np.uint8) for _ in range(5)]
        z[2][:] = 0
        z[3] = z[1].copy()
        st = _check_batch(ctx, oracle, z, 8)
        assert st["n_suffixes"] == 5 * 50001
        # tiny blocks (n <= 256 -> one starting point), 64 of them; then 65 (two runs)
        tiny = [rng.integers(97, 101, 200).astype(np.uint8) for _ in range(64)]
        _check_batch(ctx, oracle, tiny, 8)
        _check_batch(ctx, oracle, tiny + [tiny[0].copy()], 8)
        # all 256 byte values present: no code left for the sentinel -> falls back to single blocks
        full = [rng.integers(0, 256, 30000).astype(np.uint8) for _ in range(4)]
        st = _check_batch(ctx, oracle, full, 3)
        assert st["n_suffixes"] == 30001
        # unequal sizes: mixed runs
        mixed = [bw.generate("dna", n, seed=n) for n in (40000, 40000, 40000, 1000, 50000, 50000, 1, 2, 2)]
        _check_batch(ctx, oracle, mixed, 256)
        # repetitive blocks: many doubling rounds inside a batch
        rep = [np.minimum(bw.generate("repetitive", 1 << 17, seed=7 + k), 254) for k in range(4)]  # 255 byte values
        st = _check_batch(ctx, oracle, rep, 8)
        assert st["batch_blocks"] == 4 and st["rounds"] >= 3
    finally:
        ctx.close()


def test_pipeline_batches_small_blocks(oracle):
    """The pipeline groups consecutive small blocks into batches; results are delivered per block, in order."""
    sizes = [1 << 16] * 37 + [12345]
    blocks = [bw.generate("markov", n, seed=500 + i) for i, n in enumerate(sizes)]
    pipe = bw.Pipeline(1 << 16, depth=3)
    try:
        work = [x.copy() for x in blocks]
        LF, nLF, freqs, stats = pipe.run(work, 8)
        for i, x in enumerate(blocks):
            w = oracle.block(x, 8)
            assert (work[i] == w[0]).all(), i
            assert (LF[i, : nLF[i]] == w[1]).all(), i
            assert (freqs[i] == w[2]).all(), i
        assert max(s["n_suffixes"] for s in stats) > (1 << 16) + 1, "no batch was formed"
    finally:
        pipe.close()


ENGINE_KNOBS = [
    {},                                                              # defaults
    {"BWTC_RERANK_WINDOW_MB": "1"},                                  # >= 3 id windows at 1-2 MiB: bucketed rank scatter
    {"BWTC_RERANK_WINDOW_MB": "1", "BWTC_BUCKET_MIN_WINDOWS": "0"},  # one k_rerank launch per id window
    {"BWTC_RERANK_WINDOW_MB": "4", "BWTC_BUCKET_MIN_WINDOWS": "2"},  # bucketed scatter from two windows on
    {"BWTC_RERANK_WINDOW_MB": "6"},                                  # exactly two windows: one k_rerank launch per window
    {"BWTC_RERANK_WINDOW_MB": "6", "BWTC_SEG": "0"},                 # ... in doubling rounds too
    {"BWTC_RERANK_WINDOW_MB": "6", "BWTC_TWOPASS": "1"},             # exactly two windows: k_rerank + k_scatter_window (experiment, off)
    {"BWTC_RERANK_WINDOW_MB": "6", "BWTC_TWOPASS": "1", "BWTC_SEG": "0"},
    {"BWTC_RERANK_WINDOW_MB": "6", "BWTC_TWOPASS": "1", "BWTC_PACK_PRED": "0", "BWTC_AUX_MIN_MIB": "0"},
    {"BWTC_RERANK_WINDOW_MB": "6", "BWTC_HYBRID2": "1"},             # ... or window 0 direct, window 1 staged (experiment, off)
    {"BWTC_RERANK_WINDOW_MB": "6", "BWTC_HYBRID2": "1", "BWTC_SEG": "0"},  # the hybrid scatter in doubling rounds too
    {"BWTC_PACK_PRED": "0"},                                         # BWT characters gathered from the text
    {"BWTC_PACK_PRED": "0", "BWTC_AUX_MIN_MIB": "0"},                # predecessor codes as a one-byte payload array
    {"BWTC_PACK_PRED": "0", "BWTC_AUX_MIN_MIB": "0", "BWTC_RERANK_WINDOW_MB": "1"},  # ... with the bucketed scatter
    {"BWTC_STATIC_TILES": "0"},                                      # look-back kernels take tile tickets
    {"BWTC_DEBUG_FAKE_WATCHDOG": "1"},                               # watchdog fallback: retry with tickets
    {"BWTC_SEG": "0"},                                               # global radix rounds only (no segmented rounds)
    {"BWTC_SEG": "0", "BWTC_RERANK_WINDOW_MB": "1"},                 # bucketed scatter in doubling rounds too
    {"BWTC_LAZY": "0"},                                              # every rank written in round 0 (no lazy ranks)
    {"BWTC_LAZY": "2"},                                              # lazy ranks forced: singletons' ranks looked up in the sorted keys;
                                                                     # the repetitive case falls back (large groups), bit-exact either way
    {"BWTC_LAZY": "2", "BWTC_STATIC_TILES": "0"},
    {"BWTC_LAZY": "2", "BWTC_PACK_PRED": "0", "BWTC_AUX_MIN_MIB": "0"},
    {"BWTC_LAZY": "2", "BWTC_RERANK_WINDOW_MB": "1"},                # the fallback materialises ranks through the bucketed scatter
    {"BWTC_LAZY": "2", "BWTC_LADDER_FIRST": "0"},
    {"BWTC_PARTIAL": "0"},                                           # no partial character in the spare low key bits
    {"BWTC_PARTIAL": "0", "BWTC_GRAM": "0"},
    {"BWTC_GRAM": "0"},                                              # round-0 histograms counted per digit class (default: gram)
    {"BWTC_RADIX9": "1"},                                            # 9-bit digit passes where they save a pass (experiment, default off)
    {"BWTC_RADIX9": "1", "BWTC_SEG": "0"},                           # ... in the doubling rounds too
    {"BWTC_RADIX9": "1", "BWTC_SEG": "0", "BWTC_STATIC_TILES": "0"},  # ... with tile tickets
    {"BWTC_RADIX9": "1", "BWTC_PACK_PRED": "0", "BWTC_AUX_MIN_MIB": "0"},  # ... carrying the one-byte payload
]


_ORACLE_BLOCKS = {}


def _oracle_generated(oracle, kind, seed, size, x):
    """oracle.block(x, 8) of a generated input x, computed once per (kind, seed, size) for the whole module."""
    key = (kind, seed, size)
    if key not in _ORACLE_BLOCKS:
        _ORACLE_BLOCKS[key] = oracle.block(x, 8)
    return _ORACLE_BLOCKS[key]


@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()) or "default")
def test_every_engine_path_is_bit_exact(oracle, monkeypatch, knobs):
    """The engine picks between code paths by block size (L2 windows of the rank scatter, packed predecessor
    characters, segmented vs global rounds).  The tuning knobs are read when a context is created, so every path can
    be forced at sizes the oracle handles: all of them must produce the oracle's bytes.  Batches of small blocks
    (DESIGN.md §3.6) run through the same context and the same paths."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    n = (2 << 20) + 4097
    ctx = bw.CudaContext(n)
    rng = np.random.default_rng(77)
    tickets = knobs.get("BWTC_STATIC_TILES") == "0" or knobs.get("BWTC_DEBUG_FAKE_WATCHDOG") == "1"
    # (the repetitive block keeps ~all suffixes live through its global doubling rounds: with n suffixes their rank scatter
    # is windowed / bucketed exactly like round 0's)
    cases = [("markov", n), ("dna", n), ("repetitive", 1 << 20), ("repetitive", n - 5), ("random", n - 4099)]
    try:
        for kind, sz in cases:
            x = bw.generate(kind, sz, seed=41)
            if kind == "random":
                x[rng.integers(0, sz, 1000)] = 0  # zeros inside the block: the sentinel shares a code with data
            want = _oracle_generated(oracle, kind + "+zeros" if kind == "random" else kind, 41, sz, x)
            got = _gpu_block(ctx, x, 8)
            assert (got[0] == want[0]).all(), (kind, knobs)
            assert (got[1] == want[1]).all(), (kind, knobs)
            assert (got[2] == want[2]).all(), (kind, knobs)
        flags = ctx.stats()["flags"]
        if knobs.get("BWTC_LAZY") == "2":
            assert flags & 16, "lazy ranks should have been used for the last block"
        if tickets:
            assert flags & 1, "the look-back kernels should have run with ticket counters"
        else:
            assert not (flags & 1), "unexpected watchdog fallback"
        # batches: 8 x 256 KiB and a short last block fill the context (sum of n_k + 1 <= n + 1); 4 repetitive blocks keep
        # most suffixes live through global rounds
        for kind, sizes in (("markov", [1 << 18] * 8 + [4000]), ("dna", [1 << 18] * 8 + [4000]), ("repetitive", [1 << 18] * 4)):
            xs = [np.minimum(bw.generate(kind, sz, seed=60 + k), 254) for k, sz in enumerate(sizes)]  # 255 values at most
            bufs = [np.append(x, np.uint8(0xAB)) for x in xs]
            views = [b[:-1] for b in bufs]
            LF, nLF, fr = ctx.bwt_blocks(views, 8)
            st = ctx.stats()
            for k, x in enumerate(xs):
                want = _oracle_generated(oracle, kind, 60 + k, x.size, x)
                assert bufs[k][-1] == 0xAB, (kind, k, "byte after the block was written")
                assert (views[k] == want[0]).all(), (kind, k, knobs)
                assert nLF[k] == want[1].size and (LF[k, : nLF[k]] == want[1]).all(), (kind, k, knobs)
                assert (fr[k] == want[2]).all(), (kind, k, knobs)
            assert st["flags"] & 2 and st["batch_blocks"] == len(xs), (kind, st["flags"], st["batch_blocks"])
            assert not st["flags"] & (8 | 16), "a batch carries no aux payload and uses no lazy ranks"
            assert bool(st["flags"] & 1) == tickets, (kind, st["flags"])
    finally:
        ctx.close()


def _hist_chunked(a):
    h = np.zeros(256, np.int64)
    for o in range(0, a.size, 1 << 28):
        h += np.bincount(a[o:o + (1 << 28)], minlength=256)
    return h


@pytest.mark.parametrize("n", [0x40000011, 0x7FFFFFFD], ids=["just_above_2^30", "reference_limit_2^31-3"])
def test_maximum_block_size_properties(n):
    """The largest blocks: BWTC_CUDA_MAX_BLOCK = 0x7FFFFFFD bytes is the reference's own limit (blocks below 2^31 - 2,
    Compressor.cpp:78-79, PrecompressorBlock.cpp:126): N = 2^31 - 2 suffixes, 31-bit ranks, ids and look-back counts, ~86 GB of
    scratch.  No CPU checker finishes in test time at this size, so: byte histogram preserved and equal to freqs, and the
    ranks the engine reports for the sampled suffixes (LFpowers) order them exactly as a direct comparison of their
    first 64 bytes does.  The first case sits just above the 2^30 limit of the earlier 30-bit look-back words."""
    try:
        ctx = bw.CudaContext(n)
    except bw.BwtcCudaError as e:  # a smaller GPU: not this engine's target, but do not fail the suite on it
        pytest.skip(f"cannot allocate scratch for a {n >> 20} MiB block: {e}")
    x = bw.generate("random", n, seed=33)
    x[12345:12345 + 4096] = x[777:777 + 4096]  # one long repeat, so that later rounds have something to refine
    hist = _hist_chunked(x)
    blk = x.copy()
    LF = np.zeros(8, np.uint32)
    fr = np.zeros(256, np.uint32)
    pidx = ctx.bwt_block(blk, LF, fr)
    st = ctx.stats()
    ctx.close()
    assert st["n_suffixes"] == n + 1 and pidx == LF[0] and st["rounds"] >= 2
    assert (fr == hist).all() and (_hist_chunked(blk) == hist).all()
    del blk
    N = n + 1
    xs = N // 8
    pos = [0] + [N - j * xs for j in range(1, 8)]

    def suffix_prefix(p):  # first 64 bytes of suffix p of T' = reverse(X) + 0x00, without materialising T'
        idx = np.arange(p, min(p + 64, N), dtype=np.int64)
        return bytes(np.where(idx < n, x[np.minimum(n - 1 - idx, n - 1)], 0).astype(np.uint8))

    keys = [suffix_prefix(p) for p in pos]
    assert list(np.argsort(LF)) == sorted(range(8), key=lambda i: keys[i])
    assert (LF <= n).all() and len(set(LF.tolist())) == 8
    with pytest.raises(bw.BwtcCudaError):  # one byte above the limit is refused loudly (no silent truncation, no fallback)
        bw.CudaContext(0x7FFFFFFE)


def test_maximum_raw_text_size_properties():
    """The reference's largest block (2^31 - 3 bytes) reaches the raw contract (integration options A and B) as
    T = reverse(X)·0x00 of 2^31 - 2 bytes; a context of the largest capacity holds exactly that many suffixes.  The
    size-independent checks of test_maximum_block_size_properties: freqs = byte histogram of T[:-1], U keeps it (plus the
    untouched U[pidx] = T[pidx]), and the sampled suffixes' ranks order them as their first 64 bytes do."""
    N = bw.MAX_BLOCK + 1
    try:
        ctx = bw.CudaContext(bw.MAX_BLOCK)
    except bw.BwtcCudaError as e:
        pytest.skip(f"cannot allocate scratch for a {N >> 20} MiB text: {e}")
    T = np.empty(N, np.uint8)
    bw.generate("random", N - 1, seed=34, out=T)
    T[12345:12345 + 4096] = T[777:777 + 4096]
    T[-1] = 0
    hist = _hist_chunked(T[:-1])
    U = T.copy()
    LF = np.zeros(8, np.uint32)
    fr = np.zeros(256, np.uint32)
    try:
        pidx = ctx.divbwtf(U, U, LF, fr)
        st = ctx.stats()
    finally:
        ctx.close()
    assert st["n_suffixes"] == N and pidx == LF[0] and st["rounds"] >= 2
    assert U[pidx] == T[pidx]
    onehot = np.zeros(256, np.int64)
    onehot[T[pidx]] = 1
    assert (fr == hist).all() and (_hist_chunked(U) == hist + onehot).all()
    del U
    xs = N // 8
    pos = [0] + [N - j * xs for j in range(1, 8)]
    keys = [bytes(T[p:p + 64]) for p in pos]  # (a proper prefix sorts first, as bytes compare)
    assert list(np.argsort(LF)) == sorted(range(8), key=lambda i: keys[i])
    assert (LF < N).all() and len(set(LF.tolist())) == 8
