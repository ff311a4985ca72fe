"""Lazy ranks without searches (DESIGN.md §3.9): a segmented round orders the members of a group by
cmp(j) = (round-0 key of j, livebits(j) ? rank[j] + 1 : 0xFFFFFFFF) instead of by the integer rank of j.

CPU: a numpy restatement of round 0 (k_pack_round0 keys with zero padding and partial bits, the stable sort of descending
ids, a group boundary after every short suffix) and of the doubling rounds shows, for every key shape and every round the
texts reach, that doubling with cmp(i+h) gives exactly the ranks that doubling with rank(i+h) gives.
GPU: the default policy puts Markov blocks on lazy ranks and keeps the repetitive block off them, bit-exactly."""
import numpy as np
import pytest

import bwtc_b200 as bw

MiB = 1 << 20
F_LAZY, F_LAZY_ABANDONED = 16, 32


# ---- CPU restatement --------------------------------------------------------------------------------------------------
def _round0(codes, c, b, r):
    """(key, rank0, live0) of round 0.  key(i): c codes from i, then the top r bits of code c+1, zero past the end.  The
    sort is stable over descending ids, a group ends after every short suffix (its window of c (+1) codes reaches the
    end), rank = sorted position of the group head.  live0: tied after round 0, or short — the suffixes whose rank[] is
    written in lazy mode."""
    n = codes.size
    pad = np.concatenate([codes.astype(np.uint64), np.zeros(c + 2, np.uint64)])
    key = np.zeros(n, np.uint64)
    for j in range(c):
        key = (key << np.uint64(b)) | pad[j:j + n]
    if r:
        key = (key << np.uint64(r)) | (pad[c:c + n] >> np.uint64(b - r))
    ids = np.arange(n - 1, -1, -1)
    order = ids[np.argsort(key[ids], kind="stable")]
    wchars = c + (1 if r else 0)
    short = np.arange(n) >= n - wchars + 1
    sk = key[order]
    head = np.ones(n, bool)
    head[1:] = (sk[1:] != sk[:-1]) | short[order[:-1]]
    hpos = np.maximum.accumulate(np.where(head, np.arange(n), 0))
    rank = np.empty(n, np.int64)
    rank[order] = hpos
    grp = np.bincount(hpos, minlength=n)[hpos]
    live0 = np.zeros(n, bool)
    live0[order] = grp > 1
    return key, rank, live0 | short


def _double(rank, second):
    """One doubling round: sort by (rank, second), new rank = head position of the (rank, second) run."""
    n = rank.size
    order = np.lexsort((second, rank)) if second.ndim == 1 else np.lexsort((*second[::-1], rank))
    k1 = rank[order]
    k2 = second[order] if second.ndim == 1 else second[:, order]
    same = (k1[1:] == k1[:-1]) & ((k2[1:] == k2[:-1]) if k2.ndim == 1 else (k2[:, 1:] == k2[:, :-1]).all(axis=0))
    head = np.concatenate([[True], ~same])
    hpos = np.maximum.accumulate(np.where(head, np.arange(n), 0))
    out = np.empty(n, np.int64)
    out[order] = hpos
    return out


def _check_shape(codes, c, b, r):
    n = codes.size
    key, rank, live = _round0(codes, c, b, r)
    h, rounds = c, 0
    while np.unique(rank).size < n:
        idx = np.arange(n) + h
        inr = idx < n
        j = np.where(inr, idx, 0)
        full = np.where(inr, rank[j] + 1, 0)                            # the full path: rank[i+h] + 1, 0 past the end
        cmp0 = np.where(inr, key[j], np.uint64(0))                      # cmp(i+h), (0, 0) past the end
        cmp1 = np.where(inr, np.where(live[j], rank[j] + 1, 0xFFFFFFFF), 0)
        want = _double(rank, full)
        got = _double(rank, np.stack([cmp0, cmp1.astype(np.uint64)]))
        assert np.array_equal(got, want), (c, b, r, rounds)
        rank, h, rounds = want, 2 * h, rounds + 1
        assert rounds < 64
    return rounds


def _texts(rng):
    yield "iid4", rng.integers(0, 4, 3000)
    yield "iid2", rng.integers(0, 2, 2000)
    yield "markov", np.cumsum(rng.integers(0, 3, 3000)) % 7
    yield "periodic", np.tile(rng.integers(0, 5, 37), 60)
    yield "run_end", np.concatenate([rng.integers(0, 6, 1500), np.zeros(300, np.int64)])    # short suffixes tied with a run
    yield "run_end_hi", np.concatenate([rng.integers(0, 6, 1500), np.full(200, 5)])
    yield "run_mid", np.concatenate([rng.integers(1, 4, 700), np.zeros(400, np.int64), rng.integers(1, 4, 700)])
    yield "all_zero", np.zeros(700, np.int64)


@pytest.mark.parametrize("b", [1, 2, 3, 6, 8])
def test_cmp_orders_like_the_rank(b):
    """Every key shape: c from 1 to the 64-bit limit (a few), partial bits r = 0 .. b-1."""
    rng = np.random.default_rng(100 + b)
    reached = 0
    for name, t in _texts(rng):
        codes = (t % (1 << b)).astype(np.uint64)
        cmax = 64 // b
        for c in sorted({1, 2, max(1, cmax // 2), cmax - 1 if cmax > 1 else 1, cmax}):
            for r in range(0, b):
                if c * b + r > 64:
                    continue
                reached = max(reached, _check_shape(codes, c, b, r))
                wchars = c + (1 if r else 0)
                if wchars >= 2:
                    # a short suffix s and a singleton u with the same round-0 key, reached as i+h by two members of one
                    # group: ... P T 0^wchars ... P T (end), T shorter than the window
                    nz = lambda k: rng.integers(1, 1 << b, k) if b > 1 else np.ones(k, np.int64)
                    P, T = nz(40), nz(max(1, wchars // 2))
                    t = np.concatenate([nz(300), P, T, np.zeros(wchars, np.int64), nz(300), P, T])
                    reached = max(reached, _check_shape(t.astype(np.uint64), c, b, r))
    assert reached >= 3


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


@gpu
@pytest.mark.parametrize("mib", [16, 32, 64])
def test_markov_blocks_take_lazy_ranks(oracle, mib):
    """Default policy: a Markov block (memory, few repeated 8-grams) runs lazy ranks to the end, bit-exactly."""
    x = bw.generate("markov", mib * MiB, seed=71)
    ctx = bw.CudaContext(x.size)
    try:
        got = _block(ctx, x)
    finally:
        ctx.close()
    st = got[3]
    assert st["flags"] & F_LAZY and not st["flags"] & F_LAZY_ABANDONED, st["flags"]
    _assert_oracle(oracle, x, got)


@gpu
def test_repetitive_block_stays_off_lazy_ranks(oracle_record):
    """The 4 KiB-seed block repeats every 8-gram thousands of times: the policy keeps it on the full path."""
    x = bw.generate("repetitive", 16 * MiB, seed=31)
    ctx = bw.CudaContext(x.size)
    try:
        got = _block(ctx, x)
    finally:
        ctx.close()
    assert not got[3]["flags"] & F_LAZY, got[3]["flags"]
    oracle_record.check(x, 8, got[0], got[1], got[2])


@gpu
def test_divsufsort_device_exact_under_default_policy(oracle):
    import torch

    T = bw.generate("markov", 6 * MiB, seed=72)
    want, _ = oracle.suffix_array(T)
    ctx = bw.CudaContext(T.size)
    try:
        dT = torch.from_numpy(T).cuda()
        dS = torch.full((T.size,), -1, dtype=torch.int32, device="cuda")
        ctx.divsufsort_device(dT.data_ptr(), dS.data_ptr(), T.size)
        torch.cuda.synchronize()
        assert ctx.stats()["flags"] & F_LAZY
        assert np.array_equal(dS.cpu().numpy().astype(np.uint32), want)
    finally:
        ctx.close()


@gpu
def test_text_ending_in_a_run_verified(oracle, monkeypatch):
    """Short suffixes tied with live groups: a Markov block that ends in a long run of one byte, with BWTC_VERIFY=1 (every
    LFpowers entry checked on the device), against the oracle."""
    monkeypatch.setenv("BWTC_VERIFY", "1")
    x = bw.generate("markov", 8 * MiB, seed=73)
    x[-5000:] = x[-5001]
    ctx = bw.CudaContext(x.size)
    try:
        got = _block(ctx, x)
    finally:
        ctx.close()
    assert got[3]["flags"] & F_LAZY and got[3]["flags"] & bw.FLAG_VERIFIED, got[3]["flags"]
    _assert_oracle(oracle, x, got)
