"""Round 0 with digit passes over the top key digits only and the low digits sorted bucket by bucket (k_bucket_sort,
DESIGN.md §3.2): the same order as all digit passes, on every path that can take it."""
import numpy as np
import pytest

import bwtc_b200 as bw

MiB = 1 << 20
BK_CAP = 4096  # records one k_bucket_sort window holds (larger buckets take the slow path)
F_BUCKETS = bw.FLAG_ROUND0_BUCKETS
F_LAZY = 16

# extra engine settings the bucket mode must be exact under (the 8-pass mode is BWTC_ROUND0_TOP=0)
ENGINE_KNOBS = [
    {"BWTC_ROUND0_TOP": "0"},
    {"BWTC_ROUND0_TOP": "3"},
    {"BWTC_ROUND0_TOP": "4"},
    {"BWTC_ROUND0_TOP": "5"},
    {"BWTC_ROUND0_TOP": "6"},
    {"BWTC_ROUND0_TOP": "4", "BWTC_LAZY": "0"},
    {"BWTC_ROUND0_TOP": "4", "BWTC_LAZY": "2"},
    {"BWTC_ROUND0_TOP": "4", "BWTC_PACK_PRED": "0"},
    {"BWTC_ROUND0_TOP": "4", "BWTC_STATIC_TILES": "0"},
    {"BWTC_ROUND0_TOP": "4", "BWTC_DEBUG_FAKE_WATCHDOG": "1"},
    {"BWTC_ROUND0_TOP": "4", "BWTC_SEG": "0"},
]


# ---- CPU restatement ---------------------------------------------------------------------------------------------------
def _top_passes_then_buckets(keys, top):
    """Stable LSD over the top `top` 8-bit digits, then every bucket of equal top bits sorted by its low bits with ties
    in input order — what the top passes and k_bucket_sort compute."""
    low = np.uint64(64 - 8 * top)
    order = np.arange(keys.size)
    for d in range(8 - top, 8):
        digit = (keys[order] >> np.uint64(8 * d)) & np.uint64(0xFF)
        order = order[np.argsort(digit, kind="stable")]
    hi = keys[order] >> low
    heads = np.flatnonzero(np.concatenate([[True], hi[1:] != hi[:-1], [True]]))
    out = order.copy()
    for s, e in zip(heads[:-1], heads[1:]):
        seg = order[s:e]
        lowk = keys[seg] & ((np.uint64(1) << low) - np.uint64(1))
        out[s:e] = seg[np.lexsort((seg, lowk))]  # low bits, then input position
    return out


@pytest.mark.parametrize("top", [2, 3, 4, 5, 6, 7])
def test_top_passes_and_bucket_sort_give_the_full_order(top):
    rng = np.random.default_rng(top)
    for distinct in (1, 7, 300, 5000):
        base = rng.integers(0, 2**63, distinct, dtype=np.uint64) << np.uint64(1)
        keys = base[rng.integers(0, distinct, 6000)]
        keys ^= rng.integers(0, 4, keys.size, dtype=np.uint64) << np.uint64(rng.integers(0, 64))  # near ties in any digit
        want = np.lexsort((np.arange(keys.size), keys))  # all 8 stable passes: key, then input position
        assert np.array_equal(_top_passes_then_buckets(keys, top), want), (top, distinct)


# ---- GPU --------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def _block(ctx, x, starts=8):
    blk = x.copy()
    LF = np.zeros(bw.num_starting_points(x.size, starts), np.uint32)
    fr = np.zeros(256, np.uint32)
    p = ctx.bwt_block(blk, LF, fr)
    assert p == LF[0]
    return blk, LF, fr, ctx.stats()


def _assert_oracle(oracle, x, got):
    out, LF, fr = oracle.block(x, 8)
    assert np.array_equal(got[1], LF), "LFpowers"
    assert np.array_equal(got[2], fr), "freqs"
    assert np.array_equal(got[0], out), ("bytes", int(np.count_nonzero(got[0] != out)))


def _run(monkeypatch, x, top, chars=0, keybytes=0):
    monkeypatch.setenv("BWTC_ROUND0_TOP", str(top))
    ctx = bw.CudaContext(x.size)
    try:
        if chars or keybytes:
            ctx.set_round0(chars, keybytes)
        return _block(ctx, x)
    finally:
        ctx.close()


def _planted(n, g, seed):
    """A 62-symbol random text with g copies of a 21-byte string whose middle byte occurs nowhere else: the suffixes
    starting there (in either direction of the text) form one bucket of exactly g records for any top-digit count."""
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789", np.uint8)
    x = alpha[rng.integers(0, alpha.size, n)]
    pat = np.frombuffer(b"QWERTYUIOP#ASDFGHJKLZ", np.uint8)
    starts = np.sort(rng.choice(n // 32, g, replace=False)) * 32
    for s in starts:
        x[s:s + pat.size] = pat
    return x


@gpu
@pytest.mark.parametrize("mib", [16, 32])
def test_markov_blocks_take_the_bucket_sort(oracle, mib):
    """Default policy: a Markov block runs round 0 with the bucket sort, bit-exactly and with no oversized bucket."""
    x = bw.generate("markov", mib * MiB, seed=91)
    ctx = bw.CudaContext(x.size)
    try:
        got = _block(ctx, x)
    finally:
        ctx.close()
    st = got[3]
    assert st["flags"] & F_BUCKETS and st["flags"] & F_LAZY and st["round0_big_buckets"] == 0, st["flags"]
    assert st["passes"][0] < 8, st["passes"][:2]  # the top digit passes + the bucket sort
    _assert_oracle(oracle, x, got)


@gpu
def test_repetitive_and_iid_blocks_keep_every_pass(oracle):
    for kind in ("repetitive", "dna", "random"):
        x = bw.generate(kind, 4 * MiB, seed=92)
        ctx = bw.CudaContext(x.size)
        try:
            got = _block(ctx, x)
        finally:
            ctx.close()
        assert not got[3]["flags"] & F_BUCKETS, (kind, got[3]["flags"])
        _assert_oracle(oracle, x, got)


@gpu
@pytest.mark.parametrize("top", [3, 4])
@pytest.mark.parametrize("kind,chars", [("markov", 0), ("markov", 6), ("markov", 8), ("dna", 0), ("dna", 20), ("dna", 32),
                                        ("random", 8), ("random", 0)])
def test_forced_top_passes_any_key_shape(oracle, monkeypatch, top, kind, chars):
    """Every 64-bit key shape under forced top passes; 32-bit keys keep every pass.  Same bytes as the oracle."""
    n = 700001
    x = bw.generate(kind, n, seed=93)
    got = _run(monkeypatch, x, top, chars, 8 if chars else 0)
    st = got[3]
    if st["key_bytes_round0"] == 8 and -(-(st["chars_round0"] * st["bits_per_char"]) // 8) > top:
        assert st["flags"] & F_BUCKETS and st["passes"][0] == top + 1, (st["flags"], st["passes"][:2])
    else:
        assert not st["flags"] & F_BUCKETS
    _assert_oracle(oracle, x, got)


@gpu
@pytest.mark.parametrize("top", [3, 4, 5])
def test_text_ending_in_runs(oracle, monkeypatch, top):
    """Short suffixes tied with full-length keys: texts that end in runs of one byte."""
    for run in (3, 17, 5000):
        x = bw.generate("markov", 2 * MiB, seed=94 + run)
        x[-run:] = x[-run - 1]
        _assert_oracle(oracle, x, _run(monkeypatch, x, top))


@gpu
@pytest.mark.parametrize("g", [BK_CAP - 1, BK_CAP, BK_CAP + 1])
@pytest.mark.parametrize("top", [4, 6])
def test_bucket_at_the_window_capacity(oracle, monkeypatch, g, top):
    x = _planted(2 * MiB, g, seed=g)
    got = _run(monkeypatch, x, top)
    assert got[3]["flags"] & F_BUCKETS
    assert (got[3]["round0_big_buckets"] > 0) == (g > BK_CAP), got[3]["round0_big_buckets"]
    _assert_oracle(oracle, x, got)


@gpu
@pytest.mark.parametrize("top", [3, 4])
def test_one_bucket_holds_the_whole_block(oracle, monkeypatch, top):
    """A block of one byte value (plus a few others at its end): nearly every record in one oversized bucket."""
    x = np.full(3 * MiB + 5, ord("a"), np.uint8)
    x[-4:] = np.frombuffer(b"bcde", np.uint8)
    got = _run(monkeypatch, x, top)
    assert got[3]["flags"] & F_BUCKETS and got[3]["round0_big_buckets"] >= 1
    _assert_oracle(oracle, x, got)


@gpu
@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()))
def test_engine_paths(oracle, monkeypatch, knobs):
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    for seed, n in ((95, 3 * MiB + 17), (96, 4097)):
        x = bw.generate("markov", n, seed=seed)
        ctx = bw.CudaContext(x.size)
        try:
            got = _block(ctx, x)
        finally:
            ctx.close()
        if got[3]["key_bytes_round0"] == 8:  # (32-bit keys always take every pass)
            assert bool(got[3]["flags"] & F_BUCKETS) == (knobs["BWTC_ROUND0_TOP"] != "0")
        _assert_oracle(oracle, x, got)


@gpu
@pytest.mark.parametrize("top", [0, 4, 5])
def test_raw_contract_divsufsort_and_verify(oracle, monkeypatch, top):
    monkeypatch.setenv("BWTC_ROUND0_TOP", str(top))
    monkeypatch.setenv("BWTC_VERIFY", "1")
    T = bw.generate("markov", 3 * MiB + 3, seed=97)
    want_sa, _ = oracle.suffix_array(T)
    ctx = bw.CudaContext(T.size)
    try:
        got = _block(ctx, T)
        assert got[3]["flags"] & bw.FLAG_VERIFIED
        assert bool(got[3]["flags"] & F_BUCKETS) == (top != 0)
        _assert_oracle(oracle, T, got)
        sa = ctx.divsufsort(T)
        assert bool(ctx.stats()["flags"] & F_BUCKETS) == (top != 0)
        assert np.array_equal(sa.astype(np.uint32), want_sa)
        U = T.copy()  # (the raw contract leaves U[pidx] as it was)
        LF = np.zeros(8, np.uint32)
        rc = ctx.divbwtf(T, U, LF, None)
        assert bool(ctx.stats()["flags"] & F_BUCKETS) == (top != 0)
        want_rc, want_U, want_LF, _ = oracle.raw(T, 8)
        assert rc == want_rc and np.array_equal(U, want_U) and np.array_equal(LF, want_LF)
    finally:
        ctx.close()


@gpu
def test_batches_keep_every_pass(oracle, monkeypatch):
    monkeypatch.setenv("BWTC_ROUND0_TOP", "4")
    blocks = [bw.generate("markov", 1 * MiB, seed=98 + i) for i in range(4)]
    ctx = bw.CudaContext(4 * MiB + 64)
    outs = [b.copy() for b in blocks]
    try:
        LF, nLF, _ = ctx.bwt_blocks(outs, 8)
        st = ctx.stats()
    finally:
        ctx.close()
    assert st["batch_blocks"] == 4 and not st["flags"] & F_BUCKETS
    for k, (b, o) in enumerate(zip(blocks, outs)):
        want = oracle.block(b, 8)
        assert np.array_equal(o, want[0]) and np.array_equal(LF[k, :nLF[k]], want[1])
