"""GPU tests of the BATCHED forward transform (bwtc_cuda_bwt_blocks and the pipeline; DESIGN.md §3.6): a run of 2..64
equal-sized blocks (the last may be shorter) sorted as one text, with code 0 reserved for the sentinels and the block
number above the characters of every round-0 key.

Every block is compared with the C oracle (bytes, LFpowers[:nLF], nLF, freqs) from a buffer with a guard byte behind it,
and every case proves from stats() which path ran: batch flag and block count, alphabet size, code width, round-0 key
shape, packed predecessors, tile tickets.  A case that silently fell back to single blocks would check nothing.

The live counts stats() logs per round are compared with a plain reference: after ordering by the first h characters,
a suffix is live exactly when it shares its h-prefix with another suffix of its own block, i.e. when its longest common
prefix with a suffix-array neighbour in reverse(X_k) is >= h.  The LCP helper has a CPU test of its own."""
import ctypes

import numpy as np
import pytest

import bwtc_b200 as bw

GUARD = 0x5A
F_TICKETS, F_BATCH, F_PACKED, F_AUX, F_LAZY = 1, 2, 4, 8, 16


# ---- the engine's rules, restated ------------------------------------------------------------------------------------
def _ceil_log2(v):
    """Smallest b with 2^b >= v (v >= 1): ceil_log2_u64 of bwt_engine.cu."""
    return (int(v) - 1).bit_length()


def _code_bits(sigma):
    """Bits per character for an alphabet of sigma codes (a batch: the data bytes plus the reserved sentinel code)."""
    return 1 if sigma <= 2 else _ceil_log2(sigma)


def _blk_bits(nblocks):
    return max(1, _ceil_log2(nblocks))


def _forced_round0(chars, keybytes, b, blk_bits):
    """(chars_round0, key_bytes_round0) plan_round0 chooses under set_round0(chars, keybytes): the cmax64 / cmax32 rule."""
    cmax64 = (64 - blk_bits) // b
    cmax32 = 0 if blk_bits >= 32 - b else (32 - blk_bits) // b
    kb = 4 if keybytes == 4 and cmax32 >= 1 else 8
    cmax = cmax32 if kb == 4 else cmax64
    return max(1, min(chars or cmax, cmax)), kb


def _packs_pred(N, b):
    """Round 0 stores the predecessor's code above the suffix id when both fit 32 bits."""
    return max(1, _ceil_log2(N)) + b <= 32


# ---- live-count reference --------------------------------------------------------------------------------------------
def lcp_kasai(s, sa):
    """lcp[i] = length of the longest common prefix of suffixes sa[i-1] and sa[i] of s, lcp[0] = 0 (Kasai et al.).
    The comparison stops at the end of s."""
    t = np.asarray(s).tolist()
    sa = np.asarray(sa).tolist()
    n = len(t)
    rank = [0] * n
    for i, p in enumerate(sa):
        rank[p] = i
    lcp = [0] * n
    h = 0
    for i in range(n):
        r = rank[i]
        if r == 0:
            h = 0
            continue
        j = sa[r - 1]
        while i + h < n and j + h < n and t[i + h] == t[j + h]:
            h += 1
        lcp[r] = h
        if h:
            h -= 1
    return np.array(lcp, np.int64)


def max_lcp(oracle, x):
    """For every suffix of R = reverse(x) (in suffix-array order): the longest prefix it shares with another suffix of R."""
    r = np.ascontiguousarray(x[::-1])
    sa, _ = oracle.suffix_array(r)
    lcp = lcp_kasai(r, sa)
    return np.maximum(lcp, np.append(lcp[1:], 0))


def _assert_live(st, oracle, xs):
    """live[0] = N; live[r] = sum over blocks of #{suffixes whose max neighbour LCP >= prefix_len[r]} for r >= 1."""
    m = np.sort(np.concatenate([max_lcp(oracle, x) for x in xs]))
    assert st["live"][0] == st["n_suffixes"]
    for r in range(1, st["rounds"]):
        h = st["prefix_len"][r]
        want = int(m.size - np.searchsorted(m, h, side="left"))
        assert st["live"][r] == want, (r, h, st["live"], st["prefix_len"], st["passes"])


# ---- running and checking --------------------------------------------------------------------------------------------
def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


def gpu(test):
    return pytest.mark.gpu(pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")(test))


def _guarded(arrays):
    """Copies of the arrays, each a view into a buffer with one guard byte behind it."""
    bufs = []
    for a in arrays:
        b = np.empty(a.size + 1, np.uint8)
        b[:-1] = a
        b[-1] = GUARD
        bufs.append(b)
    return bufs, [b[:-1] for b in bufs]


def _check(xs, outs, LF, nLF, fr, want):
    for k, (x, w) in enumerate(zip(xs, want)):
        assert np.array_equal(np.asarray(outs[k]), w[0]), f"bytes of block {k} of {len(xs)} (n={x.size})"
        assert nLF[k] == w[1].size and np.array_equal(LF[k, : nLF[k]], w[1]), f"LFpowers of block {k} (nLF {nLF[k]})"
        assert fr is None or np.array_equal(fr[k], w[2]), f"freqs of block {k}"


def _transform(ctx, oracle, xs, starts=8, want=None):
    """bwt_blocks on guarded pageable copies of xs, checked block by block against the oracle.  Returns (stats, outputs)."""
    want = want or [oracle.block(x, starts) for x in xs]
    bufs, views = _guarded(xs)
    LF, nLF, fr = ctx.bwt_blocks(views, starts)
    st = ctx.stats()
    for k, b in enumerate(bufs):
        assert b[-1] == GUARD, f"byte after block {k} was written"
    _check(xs, views, LF, nLF, fr, want)
    return st, views


def _assert_batch(st, xs, force=None, pack_pred=True, tickets=False):
    """stats() describe ONE batch of all of xs, with the alphabet, code width, key shape and predecessor packing the
    engine's rules give for these blocks."""
    B = len(xs)
    N = sum(x.size + 1 for x in xs)
    assert st["flags"] & F_BATCH and st["batch_blocks"] == B, ("not one batch", st["flags"], st["batch_blocks"])
    assert st["n_suffixes"] == N
    sd = np.unique(np.concatenate(xs)).size
    b, blk = _code_bits(sd + 1), _blk_bits(B)
    assert st["sigma"] == sd + 1 and st["bits_per_char"] == b, (sd, st["sigma"], st["bits_per_char"])
    chars, kb = st["chars_round0"], st["key_bytes_round0"]
    assert chars >= 1 and chars * b + blk <= 8 * kb, (chars, b, blk, kb)
    if force is not None:
        assert (chars, kb) == _forced_round0(*force, b, blk), (force, b, blk, chars, kb)
    assert bool(st["flags"] & F_PACKED) == (pack_pred and _packs_pred(N, b)), (N, b, st["flags"])
    assert not st["flags"] & (F_AUX | F_LAZY), "a batch has no aux payload and no lazy ranks"
    assert bool(st["flags"] & F_TICKETS) == tickets, st["flags"]
    assert st["live"][0] == N


def _alphabet_blocks(rng, values, sizes):
    """Blocks over exactly `values`, each containing every one of them."""
    values = np.asarray(values, np.uint8)
    xs = []
    for n in sizes:
        x = rng.choice(values, n).astype(np.uint8)
        x[: values.size] = rng.permutation(values)
        xs.append(x)
    return xs


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(8 << 20)
    yield c
    c.close()


# ---- the LCP helper (CPU) --------------------------------------------------------------------------------------------
def test_lcp_helper_against_brute_force(oracle):
    rng = np.random.default_rng(1)

    def common(a, b):
        k = 0
        while k < min(a.size, b.size) and a[k] == b[k]:
            k += 1
        return k

    cases = [rng.integers(0, s, n).astype(np.uint8) for n in (1, 2, 3, 7, 40, 200) for s in (1, 2, 4, 256)]
    cases += [np.frombuffer(b"abracadabra", np.uint8).copy(), np.frombuffer(b"ab" * 30 + b"a", np.uint8).copy()]
    for s in cases:
        n = s.size
        sa, _ = oracle.suffix_array(s)
        lcp = lcp_kasai(s, sa)
        assert lcp[0] == 0
        for i in range(1, n):
            assert lcp[i] == common(s[sa[i - 1]:], s[sa[i]:]), (bytes(s), i)
        r = s[::-1].copy()
        m = np.sort(max_lcp(oracle, r))  # max_lcp reverses its argument: these are the suffixes of s
        brute = sorted(max([common(s[p:], s[q:]) for q in range(n) if q != p], default=0) for p in range(n))
        assert m.tolist() == brute, bytes(s)


# ---- 1. alphabet widths ------------------------------------------------------------------------------------------------
SIGMAS = [1, 2, 3, 4, 7, 8, 15, 16, 31, 32, 63, 64, 127, 128, 254, 255]


@gpu
@pytest.mark.parametrize("with_zero", [False, True], ids=["no0", "with0"])
@pytest.mark.parametrize("sigma", SIGMAS)
def test_alphabet_widths(ctx, oracle, sigma, with_zero):
    """Code width b = ceil(log2(sigma_data + 1)) steps at sigma_data = 2^k; 255 values is the last width before the
    fallback (8-bit codes, code 0 reserved).  0x00 as data gets a code >= 1 like any other byte."""
    rng = np.random.default_rng(100 * sigma + with_zero)
    others = rng.choice(np.arange(1, 256), sigma - 1 if with_zero else sigma, replace=False)
    values = np.concatenate([[0], others]) if with_zero else others
    for B in (3, 8):
        xs = _alphabet_blocks(rng, values, [3000] * (B - 1) + [2100])
        st, _ = _transform(ctx, oracle, xs)
        _assert_batch(st, xs)
        assert st["sigma"] == sigma + 1 and st["bits_per_char"] == max(1, _ceil_log2(sigma + 1))
        _assert_live(st, oracle, xs)


@gpu
def test_all_256_values_fall_back_to_single_blocks(ctx, oracle):
    rng = np.random.default_rng(2)
    xs = _alphabet_blocks(rng, np.arange(256), [3000] * 4 + [1000])
    st, _ = _transform(ctx, oracle, xs)
    assert st["batch_blocks"] == 1 and not st["flags"] & F_BATCH and st["n_suffixes"] == 1001


# ---- 2. block counts and full keys -------------------------------------------------------------------------------------
# chars * b + blk_bits == 64 under set_round0(0, 8): b = 1 always; b = 2 at B = 3, 4, 9, 16, 33, 63, 64 (even blk_bits);
# b = 3 at B = 2 (63 + 1) and B = 9, 16 (60 + 4).
BLOCK_COUNTS = [2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 63, 64]
ALPHABET_OF_WIDTH = {1: [0x00], 2: [0x00, 0x61, 0x62], 3: [0, 1, 2, 3, 0x41, 0x80, 0xFF], 8: list(range(200))}


@gpu
@pytest.mark.parametrize("B", BLOCK_COUNTS)
@pytest.mark.parametrize("b", sorted(ALPHABET_OF_WIDTH))
def test_block_counts_and_full_keys(ctx, oracle, b, B):
    rng = np.random.default_rng(1000 * b + B)
    values = np.array(ALPHABET_OF_WIDTH[b], np.uint8)
    xs = _alphabet_blocks(rng, values, [1500] * (B - 1) + [1000])
    want = [oracle.block(x, 8) for x in xs]
    for force in ((0, 8), (0, 4)):
        ctx.set_round0(*force)
        try:
            st, _ = _transform(ctx, oracle, xs, want=want)
        finally:
            ctx.set_round0(0, 0)
        _assert_batch(st, xs, force=force)
        assert st["bits_per_char"] == b and st["batch_blocks"] == B
        _assert_live(st, oracle, xs)


@gpu
def test_65_blocks_and_an_unbatched_context(ctx, oracle, monkeypatch):
    """65 blocks: a run of 64, then one on its own; a context with BWTC_BATCH=0 transforms every block alone.  The bytes
    are identical either way."""
    rng = np.random.default_rng(3)
    xs = [rng.integers(0, 5, 2000).astype(np.uint8) for _ in range(65)]
    want = [oracle.block(x, 8) for x in xs]
    st, run64 = _transform(ctx, oracle, xs[:64], want=want[:64])
    _assert_batch(st, xs[:64])
    st, all65 = _transform(ctx, oracle, xs, want=want)
    assert st["batch_blocks"] == 1 and st["n_suffixes"] == 2001 and not st["flags"] & F_BATCH
    monkeypatch.setenv("BWTC_BATCH", "0")
    c0 = bw.CudaContext(8 << 20)
    try:
        st, single = _transform(c0, oracle, xs, want=want)
    finally:
        c0.close()
    assert st["batch_blocks"] == 1 and not st["flags"] & F_BATCH
    for k in range(65):
        assert np.array_equal(all65[k], single[k]) and (k == 64 or np.array_equal(run64[k], single[k])), k


# ---- 3. forced key shapes: many doubling rounds inside a batch -------------------------------------------------------
def _kind_blocks(kind, sizes, seed):
    xs = []
    for k, n in enumerate(sizes):
        r = np.random.default_rng(seed + k)
        if kind == "zeros":
            x = np.zeros(n, np.uint8)
            x[r.integers(0, n, n // 100)] = r.integers(1, 4, n // 100)
        elif kind == "tiled":  # a 300-byte period with rare mutations: hundreds of suffixes share every short prefix
            x = np.resize(r.integers(1, 255, 300).astype(np.uint8), n)
            x[r.integers(0, n, n // 1000)] = r.integers(1, 255, n // 1000)
        elif kind == "planted":  # i.i.d. bytes and one 200-byte segment repeated: only the copies stay live after round 0
            x = r.integers(1, 255, n).astype(np.uint8)
            x[n // 2:n // 2 + 200] = x[1000:1200]
        else:
            x = bw.generate(kind, n, seed=seed + k)
            if kind == "repetitive":  # (its bytes take all 256 values, which a batch cannot hold: 0xFF -> 0xFE)
                x = np.minimum(x, 254)
        xs.append(x)
    return xs


@gpu
@pytest.mark.parametrize("force", [(1, 4), (2, 4), (3, 4), (1, 8), (5, 8), (64, 8)])
@pytest.mark.parametrize("kind", ["markov", "dna", "repetitive", "zeros"])
def test_forced_key_shapes_in_a_batch(ctx, oracle, kind, force):
    """A short round-0 key sends the batch through global radix rounds, segmented rounds and the tail: a live suffix must
    never read rank[i + h] of another block."""
    xs = _kind_blocks(kind, [1 << 15] * 5 + [20001], seed=40)
    ctx.set_round0(*force)
    try:
        st, _ = _transform(ctx, oracle, xs)
    finally:
        ctx.set_round0(0, 0)
    _assert_batch(st, xs, force=force)
    if st["chars_round0"] <= 5:
        assert st["rounds"] >= 3, ("doubling rounds expected", st["rounds"], st["live"])
    assert all(a < b for a, b in zip(st["prefix_len"][1:], st["prefix_len"][2:])), st["prefix_len"]
    if st["rounds"] > 1:
        assert st["prefix_len"][1] == st["chars_round0"]
    _assert_live(st, oracle, xs)


# ---- 4. (engine paths: tests/test_gpu_parity.py::test_every_engine_path_is_bit_exact has a batched leg) -----------------

# ---- 5. predecessor packing ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n0,packed", [((1 << 20) - 1, True), (1 << 20, False)], ids=["N=2^24", "N=2^24+16"])
def test_predecessor_packing_boundary(oracle, n0, packed):
    """8-bit codes (251 byte values): ceil(log2 N) + 8 <= 32 holds up to N_total = 2^24.  16 x (2^20 - 1) bytes are exactly
    2^24 suffixes (codes packed above the ids); 16 x 2^20 bytes are 2^24 + 16 (BWT bytes gathered from the text, block
    starts found by owns_hole)."""
    xs = [bw.generate("random", n0, seed=50 + k) % 251 for k in range(16)]
    assert np.unique(np.concatenate(xs)).size == 251
    c = bw.CudaContext((1 << 24) + 64)
    try:
        st, _ = _transform(c, oracle, xs)
    finally:
        c.close()
    _assert_batch(st, xs)
    assert st["bits_per_char"] == 8 and bool(st["flags"] & F_PACKED) == packed


@gpu
def test_pack_pred_off(oracle, monkeypatch):
    monkeypatch.setenv("BWTC_PACK_PRED", "0")
    xs = _kind_blocks("markov", [20000] * 5 + [7777], seed=60)
    xs[2][::97] = 0
    c = bw.CudaContext(1 << 20)
    try:
        st, _ = _transform(c, oracle, xs)
    finally:
        c.close()
    _assert_batch(st, xs, pack_pred=False)
    _assert_live(st, oracle, xs)


# ---- 6. buffers and bookkeeping --------------------------------------------------------------------------------------
def _pinned_guarded(xs):
    import torch

    ts = []
    for x in xs:
        t = torch.empty(x.size + 1, dtype=torch.uint8).pin_memory()
        a = t.numpy()
        a[:-1] = x
        a[-1] = GUARD
        ts.append(t)
    return ts, [t.numpy()[:-1] for t in ts]


def _buffer_blocks():
    return _kind_blocks("markov", [40000] * 6 + [17000], seed=70)


@gpu
def test_buffer_kinds_through_bwt_blocks(ctx, oracle):
    """Pinned, pageable, mixed (the copy kind is chosen from block 0's buffer) and in-place device blocks."""
    import torch

    xs = _buffer_blocks()
    want = [oracle.block(x, 8) for x in xs]
    half = len(xs) // 2
    pin_ts, pin_views = _pinned_guarded(xs)
    pg_bufs, pg_views = _guarded(xs)
    layouts = {"pinned": pin_views, "pinned_then_pageable": pin_views[:half] + pg_views[half:],
               "pageable_then_pinned": pg_views[:half] + pin_views[half:]}
    for name, views in layouts.items():
        for v, x in zip(views, xs):
            v[:] = x
        LF, nLF, fr = ctx.bwt_blocks(views, 8)
        st = ctx.stats()
        _assert_batch(st, xs)
        _check(xs, views, LF, nLF, fr, want)
        for t in pin_ts:
            assert t.numpy()[-1] == GUARD, name
        for b in pg_bufs:
            assert b[-1] == GUARD, name
    dev = [torch.from_numpy(np.append(x, np.uint8(GUARD))).cuda() for x in xs]
    LF, nLF, fr = ctx.bwt_blocks([(t.data_ptr(), x.size) for t, x in zip(dev, xs)], 8, on_device=True)
    torch.cuda.synchronize()
    _assert_batch(ctx.stats(), xs)
    host = [t.cpu().numpy() for t in dev]
    assert all(h[-1] == GUARD for h in host)
    _check(xs, [h[:-1] for h in host], LF, nLF, fr, want)


@gpu
def test_buffer_kinds_through_the_pipeline(oracle):
    """Pipeline.run_ptrs with separate inputs and outputs (host pageable, pinned, both mixes; device): the outputs are
    right, the guards and the inputs untouched."""
    import torch

    xs = _buffer_blocks()
    want = [oracle.block(x, 8) for x in xs]
    half = len(xs) // 2
    p = bw.Pipeline(40000, depth=2)
    try:
        pin_ts, pin_views = _pinned_guarded([np.zeros_like(x) for x in xs])
        pg_bufs, pg_views = _guarded([np.zeros_like(x) for x in xs])
        in_pin_ts, in_pin = _pinned_guarded(xs)
        in_pg = [x.copy() for x in xs]
        layouts = {"pageable": (in_pg, pg_views), "pinned": (in_pin, pin_views),
                   "pinned_then_pageable": (in_pin[:half] + in_pg[half:], pin_views[:half] + pg_views[half:]),
                   "pageable_then_pinned": (in_pg[:half] + in_pin[half:], pg_views[:half] + pin_views[half:])}
        for name, (ins, outs) in layouts.items():
            for o in outs:
                o[:] = 0
            LF, nLF, fr, stats = p.run_ptrs([a.ctypes.data for a in ins], [o.ctypes.data for o in outs],
                                            [x.size for x in xs], 8, on_device=False)
            for s in stats:
                _assert_batch(s, xs)
            _check(xs, outs, LF, nLF, fr, want)
            for a, x in zip(ins, xs):
                assert np.array_equal(a, x), (name, "input changed")
            assert all(t.numpy()[-1] == GUARD for t in pin_ts) and all(b[-1] == GUARD for b in pg_bufs), name
        din = [torch.from_numpy(x.copy()).cuda() for x in xs]
        dout = [torch.full((x.size + 1,), GUARD, dtype=torch.uint8, device="cuda") for x in xs]
        LF, nLF, fr, stats = p.run_ptrs([t.data_ptr() for t in din], [t.data_ptr() for t in dout], [x.size for x in xs], 8,
                                        on_device=True)
        torch.cuda.synchronize()
        for s in stats:
            _assert_batch(s, xs)
        host = [t.cpu().numpy() for t in dout]
        assert all(h[-1] == GUARD for h in host)
        _check(xs, [h[:-1] for h in host], LF, nLF, fr, want)
        for t, x in zip(din, xs):
            assert np.array_equal(t.cpu().numpy(), x)
    finally:
        p.close()


@gpu
@pytest.mark.parametrize("n0", [1, 2, 3])
def test_tiny_blocks(ctx, oracle, n0):
    rng = np.random.default_rng(n0)
    for B in (2, 5, 64):
        for n_last in range(1, n0 + 1):
            xs = [rng.integers(0, 3, n0).astype(np.uint8) for _ in range(B - 1)] + [rng.integers(0, 3, n_last).astype(np.uint8)]
            st, _ = _transform(ctx, oracle, xs, starts=8)
            _assert_batch(st, xs)
            _assert_live(st, oracle, xs)


@gpu
@pytest.mark.parametrize("starts", [1, 7, 8, 256])
@pytest.mark.parametrize("n_last", [1, 255, 256, 257, 999, 1000])
def test_last_block_bookkeeping(ctx, oracle, n_last, starts):
    """nLF of the last block differs from the others when n_last <= 256 < n0 (one starting point)."""
    rng = np.random.default_rng(n_last * 1000 + starts)
    xs = [rng.integers(0, 6, 1000).astype(np.uint8) for _ in range(5)] + [rng.integers(0, 6, n_last).astype(np.uint8)]
    bufs, views = _guarded(xs)
    LF, nLF, fr = ctx.bwt_blocks(views, starts)
    st = ctx.stats()
    _assert_batch(st, xs)
    assert all(b[-1] == GUARD for b in bufs)
    assert list(nLF) == [bw.num_starting_points(x.size, starts) for x in xs]
    _check(xs, views, LF, nLF, fr, [oracle.block(x, starts) for x in xs])
    assert not LF[-1, nLF[-1]:].any() and not LF[0, nLF[0]:].any(), "LFpowers rows written past nLF"


@gpu
def test_freqs_rows_are_incremented(ctx, oracle):
    rng = np.random.default_rng(9)
    xs = _kind_blocks("dna", [30000] * 4 + [12345], seed=80)
    B = len(xs)
    bufs, views = _guarded(xs)
    ptrs = (ctypes.c_void_p * B)(*[v.ctypes.data for v in views])
    sizes = np.array([x.size for x in xs], np.uint32)
    LF = np.zeros((B, 256), np.uint32)
    nLF = np.zeros(B, np.uint32)
    fr0 = rng.permutation(B * 256).reshape(B, 256).astype(np.uint32) + 1  # distinct, non-zero
    fr = fr0.copy()
    ctx._check(ctx._lib.bwtc_cuda_bwt_blocks(ctx._h, ptrs, sizes.ctypes.data, B, 8, 0, LF.ctypes.data, nLF.ctypes.data,
                                             fr.ctypes.data))
    _assert_batch(ctx.stats(), xs)
    want = [oracle.block(x, 8) for x in xs]
    _check(xs, views, LF, nLF, None, want)
    for k, x in enumerate(xs):
        assert np.array_equal(fr[k], fr0[k] + np.bincount(x, minlength=256).astype(np.uint32)), k
        assert np.array_equal(fr[k] - fr0[k], want[k][2]), k


@gpu
@pytest.mark.parametrize("B", [2, 5])
def test_capacity_exactly_full_and_one_over(oracle, B):
    """A run is batched while sum(n_k + 1) <= capacity + 1; one byte more and the blocks go one by one, same bytes."""
    xs = _kind_blocks("markov", [3000] * (B - 1) + [2222], seed=90)
    total = sum(x.size + 1 for x in xs)
    want = [oracle.block(x, 8) for x in xs]
    outs = {}
    for cap, batched in ((total - 1, True), (total - 2, False)):
        c = bw.CudaContext(cap)
        try:
            st, outs[batched] = _transform(c, oracle, xs, want=want)
        finally:
            c.close()
        if batched:
            _assert_batch(st, xs)
        else:
            assert st["batch_blocks"] == 1 and not st["flags"] & F_BATCH and st["n_suffixes"] == xs[-1].size + 1
    for a, b in zip(outs[True], outs[False]):
        assert np.array_equal(a, b)


# ---- 7. live counts against the reference --------------------------------------------------------------------------
SMALL_MAX = 2048  # bwt_kernels.cuh: the tail kernel takes over at this many live suffixes; segmented rounds run above it


def _entry_kinds(st):
    """What logged the entries r >= 1: a global radix round (digit passes), a segmented round (sort-free, more than
    SMALL_MAX live) or the tail (k_small_rounds: at most SMALL_MAX live, all remaining rounds in one entry)."""
    return ["global" if st["passes"][r] else ("segmented" if st["live"][r] > SMALL_MAX else "tail")
            for r in range(1, st["rounds"])]


@gpu
def test_live_counts_of_batches(ctx, oracle):
    """The reference holds for every kind of logged entry, and all three kinds appear among these inputs.  The generated
    repetitive blocks (period 4096) leave groups of ~32 after round 0, within the segmented rounds' limit of 128; a
    300-byte period leaves groups of hundreds, which need global radix rounds first.  Periodic blocks stay live until h
    passes the repeat length and then drop to 0 at once; Markov and DNA blocks of this size finish in one segmented round.
    The tail (at most SMALL_MAX live, not yet 0) comes from i.i.d. blocks with one planted repeat: after round 0 only the
    ~400 suffixes in its two copies per block are live."""
    seen = {}
    for kind, needs in (("markov", ()), ("dna", ()), ("repetitive", ("segmented",)), ("tiled", ("global",)),
                        ("planted", ("tail",))):
        xs = _kind_blocks(kind, [1 << 17] * 3 + [100003], seed=110)
        st, _ = _transform(ctx, oracle, xs)
        _assert_batch(st, xs)
        _assert_live(st, oracle, xs)
        kinds = _entry_kinds(st)
        seen[kind] = kinds
        for e in needs:
            assert e in kinds, (kind, e, kinds, st["live"])
    assert {"global", "segmented", "tail"} <= {e for k in seen.values() for e in k}, seen


@gpu
@pytest.mark.parametrize("kind", ["markov", "dna", "repetitive"])
def test_live_counts_of_single_blocks(oracle, monkeypatch, kind):
    """Without the partial character (BWTC_PARTIAL=0) and without 0x00 in the block (the sentinel is then outside the
    alphabet), round 0 orders exactly chars_round0 characters, so the same reference applies to a single block."""
    monkeypatch.setenv("BWTC_PARTIAL", "0")
    x = bw.generate(kind, 1 << 17, seed=120)
    x[x == 0] = 1
    c = bw.CudaContext(x.size)
    try:
        st, _ = _transform(c, oracle, [x])
    finally:
        c.close()
    assert not st["flags"] & F_BATCH and st["n_suffixes"] == x.size + 1 and st["rounds"] >= 2
    _assert_live(st, oracle, [x])
