"""GPU tests of the single-block INVERSE transform (bwtc_cuda_inverse_block, _device, _raw, and bwtc_cuda_inverse_blocks
with one block; run_inverse in bwt_engine.cu, kernels in ibwt_kernels.cuh) at the edges its kernels depend on:
- the splitter geometry: spacing K = 32, S0 = ceil(N / 32) splitters, ceil(log2 S0) pointer-jumping rounds, 256-thread
  walk CTAs;
- the end-of-block row (eob) at 1, at N - 1 and on a splitter;
- the 9-bit keys (byte 0x00 is key 1, byte 0xFF key 256, which shares low digit 0 with the end-of-block row's key 0);
- every buffer kind and entry point, under every engine path, including a faked look-back watchdog whose retry must start
  from the device copy of the input, because the speculative copy may already have overwritten a pinned in-place block;
- the capacity edge, the scratch the inverse borrows from the forward transform, and the largest block.

The reference is the block x itself, and oracle.inverse_block (the restatement of the reference's inverse) on the oracle's
forward output.  Every host buffer carries a guard byte after the block that must survive; inverse_raw must leave its
last row L[N-1] as it was."""
import itertools

import numpy as np
import pytest

import bwtc_b200 as bw


def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")]

GUARD = 0x5A
INV_K = 32  # splitter spacing of the inverse (BWTC_INV_K)


def _jump_rounds(N):
    """ceil(log2 S0) pointer-jumping rounds over S0 = ceil(N / 32) splitters."""
    return (-(-N // INV_K) - 1).bit_length()


def _ref(oracle, x, starts=1):
    """The oracle's forward output of x and its end-of-block row; the oracle's inverse must restore x."""
    b, LF, _ = oracle.block(x, starts)
    eob = int(LF[0])
    assert np.array_equal(oracle.inverse_block(b, eob), x)
    return b, eob


def _raw(b, eob, hole):
    """The raw form (N = n + 1 rows) of a block-contract output: the byte moved into the hole goes back to row N - 1 (as
    InverseBWT.cpp:49 does) and the end-of-block row, which the inverse ignores, is set to `hole`."""
    n = b.size
    raw = np.empty(n + 1, np.uint8)
    raw[:n] = b
    raw[n] = b[eob] if eob < n else 0  # (eob = N - 1: nothing was moved)
    raw[eob] = hole
    return raw


def _host(a, pinned):
    """A copy of a followed by one guard byte, in pageable or pinned host memory."""
    if pinned:
        import torch

        buf = torch.empty(a.size + 1, dtype=torch.uint8).pin_memory().numpy()
    else:
        buf = np.empty(a.size + 1, np.uint8)
    buf[:-1] = a
    buf[-1] = GUARD
    return buf


def _dev(a):
    import torch

    d = torch.empty(a.size + 1, dtype=torch.uint8, device="cuda")
    d[:-1] = torch.from_numpy(a)
    d[-1] = GUARD
    return d


# (entry point, buffer kind, in place)
WAYS = ["block-pageable", "block-pinned", "device-inplace", "device-out", "raw-pageable", "raw-pinned",
        "blocks-pageable-inplace", "blocks-pinned-inplace", "blocks-device-inplace",
        "blocks-pageable-out", "blocks-pinned-out", "blocks-device-out"]


def _invert(ctx, way, b, eob, hole=0xEE):
    """Restores the block-contract output b (end-of-block row eob) through one entry point and buffer kind.  Checks the
    guard bytes, that a separate input is not written and that raw row N - 1 stays as it was; returns the restored bytes
    and the call's stats."""
    import torch

    n = b.size
    row = np.array([eob], np.uint32)
    if way.startswith("block-"):
        buf = _host(b, way == "block-pinned")
        assert ctx.inverse_block(buf[:-1], row) == n
        assert buf[-1] == GUARD, "byte after the block was written"
        return buf[:-1].copy(), ctx.stats()
    if way.startswith("raw-"):
        raw = _raw(b, eob, hole)
        buf = _host(raw, way == "raw-pinned")
        assert ctx.inverse_raw(buf[:-1], row) == n
        assert buf[n] == raw[n] and buf[-1] == GUARD, "raw row N - 1 or the byte after it was written"
        return buf[:n].copy(), ctx.stats()
    if way.startswith("device-"):
        d = _dev(b)
        out = d if way == "device-inplace" else _dev(np.full(n, 0xC3, np.uint8))
        assert ctx.inverse_block_device(d.data_ptr(), out.data_ptr(), n, eob) == n
        torch.cuda.synchronize()
        o = out.cpu().numpy()
        assert o[-1] == GUARD, "byte after the device output was written"
        if out is not d:
            assert np.array_equal(d.cpu().numpy()[:-1], b), "the separate device input was written"
        return o[:-1].copy(), ctx.stats()
    _, kind, place = way.split("-")
    if kind == "device":
        src = _dev(b)
        dst = src if place == "inplace" else _dev(np.full(n, 0xC3, np.uint8))
        ctx.inverse_blocks([(src.data_ptr(), n)], [row], on_device=True,
                           out=None if place == "inplace" else [(dst.data_ptr(), n)])
        torch.cuda.synchronize()
        s, o = src.cpu().numpy(), dst.cpu().numpy()
    else:
        s = _host(b, kind == "pinned")
        o = s if place == "inplace" else _host(np.full(n, 0xC3, np.uint8), kind == "pinned")
        ctx.inverse_blocks([s[:-1]], [row], out=None if place == "inplace" else [o[:-1]])
    assert o[-1] == GUARD and s[-1] == GUARD, "byte after the block was written"
    if place == "out":
        assert np.array_equal(s[:-1], b), "the separate input was written"
    return o[:-1].copy(), ctx.stats()


def _check_stats(st, N, tickets):
    assert st["n_suffixes"] == N and st["batch_blocks"] == 1
    assert not st["flags"] & bw.FLAG_CORRUPT, "a valid block was flagged corrupt"
    assert not st["flags"] & 2, "one block must not take the batch path"
    assert bool(st["flags"] & 1) == tickets, ("ticket flag", st["flags"], tickets)
    assert st["rounds"] == _jump_rounds(N), (st["rounds"], N)


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(4 << 20)
    yield c
    c.close()


# ---- tiny blocks: one splitter, no jump rounds, every end-of-block row ---------------------------------------------

@pytest.mark.parametrize("alphabet,top", [((0x00, 0xFF), 11), ((0x00, 0x80, 0xFF), 7)], ids=["binary", "ternary"])
def test_every_tiny_text(ctx, oracle, alphabet, top):
    """Every text of 1..11 bytes over {0x00, 0xFF} and of 1..7 bytes over {0x00, 0x80, 0xFF}: the byte values at both ends
    of the key range, and between them every end-of-block row 1..n a text of that length can have."""
    for n in range(1, top + 1):
        eobs = set()
        for t in itertools.product(alphabet, repeat=n):
            x = np.array(t, np.uint8)
            b, eob = _ref(oracle, x)
            eobs.add(eob)
            buf = _host(b, False)
            assert ctx.inverse_block(buf[:-1], np.array([eob], np.uint32)) == n
            assert buf[-1] == GUARD and np.array_equal(buf[:-1], x), (n, t, eob)
        assert eobs == set(range(1, n + 1)), (n, sorted(eobs))
        assert ctx.stats()["rounds"] == 0


# ---- splitter geometry -----------------------------------------------------------------------------------------------

def _geometry_inputs(n, seed):
    rng = np.random.default_rng(seed)
    xs = [rng.integers(0, s, n).astype(np.uint8) for s in (1, 2, 4, 256)]
    for p in (31, 32, 33, 64):  # periods that line up with the splitter spacing
        xs.append(np.tile(rng.integers(0, 256, p).astype(np.uint8), n // p + 1)[:n])
    return xs


def _check_geometry(ctx, oracle, Ns, seed):
    for N in Ns:
        n = N - 1
        for i, x in enumerate(_geometry_inputs(n, seed + N)):
            if N <= 32 * (1 << 15) + 1:
                b, eob = _ref(oracle, x)
            else:  # the GPU forward (oracle-checked at these sizes elsewhere); the inverse must give x back
                b = x.copy()
                LF = np.zeros(1, np.uint32)
                ctx.bwt_block(b, LF, None)
                eob = int(LF[0])
            buf = _host(b, False)
            assert ctx.inverse_block(buf[:-1], np.array([eob], np.uint32)) == n
            assert buf[-1] == GUARD, (N, i)
            assert np.array_equal(buf[:-1], x), f"N = {N} (S0 = {-(-N // INV_K)}), input {i} not restored"
            st = ctx.stats()
            assert st["n_suffixes"] == N and st["rounds"] == _jump_rounds(N), (N, st["rounds"])


@pytest.mark.parametrize("r", range(18))
def test_splitter_counts_around_powers_of_two(ctx, oracle, r):
    """N = 32 * 2^r and 32 * 2^r + 1 rows: S0 = 2^r and 2^r + 1 splitters, so every jump-round count is met exactly at
    its edge, and r = 8 straddles one and two 256-splitter walk CTAs."""
    _check_geometry(ctx, oracle, (32 << r, (32 << r) + 1), 100 + r)


def test_block_sizes_around_the_splitter_spacing(ctx, oracle):
    _check_geometry(ctx, oracle, [32 * k + d for k in (1, 2, 3) for d in (-1, 0, 1)], 200)


# ---- end-of-block row placed on purpose -------------------------------------------------------------------------------

def _eob_one(n, hole, rng):
    """X[n-1] the unique minimum (end-of-block row 1); the largest suffix of T' = reverse(X).$ starts at the unique
    maximum 0xFF, so the byte moved into the hole, L[N-1], is the byte after it in X."""
    x = rng.integers(1, 0xFF, n).astype(np.uint8)
    x[-1] = 0x00
    i = n - 2 if hole == 0x00 else int(rng.integers(0, n - 2))
    x[i] = 0xFF
    x[i + 1] = hole
    return x


def _eob_on_splitter(n, hole, seed):
    """Searches seeds for a text whose end-of-block row is a multiple of 32: the stretch of splitter 0 (the sentinel row)
    then ends after one step.  The byte moved into the hole is `hole` (as in _eob_one)."""
    for s in itertools.count(seed):
        rng = np.random.default_rng(s)
        x = rng.integers(1, 0xFF, n).astype(np.uint8)
        i = int(rng.integers(0, n - 1))
        x[i] = 0xFF
        x[i + 1] = hole
        yield x


EOB_SIZES = [2, 3, 31, 32, 33, 63, 64, 65, 1000, 8191, 8192, 8193, 300001]


@pytest.mark.parametrize("hole", [0x00, 0xFE], ids=["hole00", "holeFE"])
def test_end_of_block_row_one(ctx, oracle, hole):
    """eob = 1.  L[N-1] cannot be 0xFF in any BWT (0xFF.s > s for the largest suffix s, so 0xFF never precedes it), so
    the largest value the moved byte can take is 0xFE; raw inputs also get 0x00 and 0xFF in the ignored row."""
    rng = np.random.default_rng(300 + hole)
    for n in EOB_SIZES[hole != 0x00:]:
        x = _eob_one(n, hole, rng)
        b, eob = _ref(oracle, x)
        assert eob == 1 and b[eob] == hole, (n, eob, b[eob])
        for way in WAYS:
            for raw_hole in ((0x00, 0xFF) if way.startswith("raw") else (0xEE,)):
                got, _ = _invert(ctx, way, b, eob, raw_hole)
                assert np.array_equal(got, x), (n, way, raw_hole)


@pytest.mark.parametrize("kind", ["unique_max", "all_00", "all_FF"])
def test_end_of_block_row_last(ctx, oracle, kind):
    """eob = N - 1: the end-of-block row is the last row itself, so in block mode no byte was moved into the hole."""
    rng = np.random.default_rng(400)
    for n in [1] + EOB_SIZES:
        if kind == "unique_max":
            x = rng.integers(0, 0xFF, n).astype(np.uint8)
            x[-1] = 0xFF
        else:
            x = np.full(n, 0x00 if kind == "all_00" else 0xFF, np.uint8)
        b, eob = _ref(oracle, x)
        assert eob == n, (n, eob)
        for way in WAYS:
            for raw_hole in ((0x00, 0xFF) if way.startswith("raw") else (0xEE,)):
                got, _ = _invert(ctx, way, b, eob, raw_hole)
                assert np.array_equal(got, x), (n, way, raw_hole)


@pytest.mark.parametrize("hole", [0x00, 0xFE], ids=["hole00", "holeFE"])
def test_end_of_block_row_on_a_splitter(ctx, oracle, hole):
    for n in (64, 1000, 4097, 100000):
        for x in _eob_on_splitter(n, hole, 500 + n):
            b, eob = _ref(oracle, x)
            if eob % INV_K == 0:
                break
        assert eob >= INV_K and b[eob] == hole, (n, eob, b[eob])
        for way in WAYS:
            for raw_hole in ((0x00, 0xFF) if way.startswith("raw") else (0xEE,)):
                got, _ = _invert(ctx, way, b, eob, raw_hole)
                assert np.array_equal(got, x), (n, eob, way, raw_hole)


# ---- the 9-bit key's byte edges ---------------------------------------------------------------------------------------

def _byte_edge_blocks(n, rng):
    all256 = rng.integers(0, 256, n).astype(np.uint8)
    all256[rng.permutation(n)[: min(n, 256)]] = np.arange(min(n, 256), dtype=np.uint8)
    heavy = np.full(n, 0xFF, np.uint8)  # key 256 (low digit 0) far outnumbers everything else
    heavy[rng.random(n) < 0.03] = 0x00
    heavy[rng.random(n) < 0.01] = 0x01
    return {"only00": np.zeros(n, np.uint8), "onlyFF": np.full(n, 0xFF, np.uint8),
            "00_FF": np.where(rng.random(n) < 0.5, 0x00, 0xFF).astype(np.uint8), "all256": all256, "FF_heavy": heavy}


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 255, 256, 257, 4096, 65537, (1 << 20) + 3])
def test_key_byte_edges(ctx, oracle, n):
    rng = np.random.default_rng(600 + n)
    for name, x in _byte_edge_blocks(n, rng).items():
        b, eob = _ref(oracle, x, 8)
        for way in WAYS:
            got, st = _invert(ctx, way, b, eob)
            assert np.array_equal(got, x), (name, n, way)
            assert st["n_suffixes"] == n + 1 and not st["flags"] & bw.FLAG_CORRUPT


# ---- buffer kinds x entry points x engine paths ---------------------------------------------------------------------

PATHS = {
    "default": {},
    "tickets": {"BWTC_STATIC_TILES": "0"},
    "fake_watchdog": {"BWTC_DEBUG_FAKE_WATCHDOG": "1"},
    "wait0": {"BWTC_WAIT_MODE": "0"},
    "wait1": {"BWTC_WAIT_MODE": "1"},
    "wait2": {"BWTC_WAIT_MODE": "2"},
}
CAP = 2 << 20


def _path_inputs():
    return [bw.generate("markov", (1 << 20) + 13, seed=700), bw.generate("random", 70001, seed=701),
            bw.generate("dna", 33, seed=702), _byte_edge_blocks(4097, np.random.default_rng(703))["FF_heavy"]]


def _stale_out_ctx(y):
    """A fresh context (with this test's knobs) created right after a context of the same capacity transformed and
    restored y, a block other than the one under test, and was closed: the new context's output scratch holds bytes of
    y or fresh memory, so what the speculative copy moves after a faked watchdog is really stale (after a forward of the
    block under test it would hold the very bytes that are to be inverted)."""
    c = bw.CudaContext(CAP)
    try:
        b = y.copy()
        LF = np.zeros(1, np.uint32)
        c.bwt_block(b, LF, None)
        c.inverse_block(b, LF)
        assert np.array_equal(b, y)
    finally:
        c.close()
    return bw.CudaContext(CAP)


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("way", WAYS)
def test_engine_paths(oracle, monkeypatch, path, way):
    """Each entry point and buffer kind under default knobs, ticket tile ids, a faked look-back watchdog in the inverse's
    digit passes, and each host wait mode.  The faked watchdog leaves what a real one leaves (walk1, jump and walk2 return
    at entry; the speculative pinned copy moves stale bytes), and the retry with ticket tile ids must restore the block
    from the device copy of the input.  It fires once per context, so every block gets a fresh context."""
    for k, v in PATHS[path].items():
        monkeypatch.setenv(k, v)
    fake = path == "fake_watchdog"
    tickets = path in ("tickets", "fake_watchdog")
    xs = _path_inputs()
    refs = [_ref(oracle, x, 8) for x in xs]
    c = None if fake else bw.CudaContext(CAP)
    try:
        for i, (x, (b, eob)) in enumerate(zip(xs, refs)):
            if fake:
                c = _stale_out_ctx(bw.generate("random", x.size, seed=710 + i))
            got, st = _invert(c, way, b, eob, hole=0x00 if i % 2 else 0xFF)
            assert np.array_equal(got, x), (path, way, i)
            _check_stats(st, x.size + 1, tickets)
            if fake:
                c.close()
    finally:
        if c is not None:
            c.close()


# ---- capacity edge and refused arguments ------------------------------------------------------------------------------

def _refused(call, *bufs):
    before = [np.array(b, copy=True) for b in bufs]
    with pytest.raises(bw.BwtcCudaError) as e:
        call()
    for b0, b in zip(before, bufs):
        assert np.array_equal(b0, b), "a refused call wrote into a buffer"
    return e.value.code


def test_capacity_edge_and_refused_arguments(oracle):
    import torch

    """On a context of capacity m: an inverse block of m bytes and a raw input of m + 1 rows are accepted, one byte more
    is refused with ETOOBIG; empty inputs and end-of-block rows outside [0, N) are refused with EARG.  A refused call
    writes nothing."""
    m = 100003
    c = bw.CudaContext(m)
    try:
        rng = np.random.default_rng(800)
        x = rng.integers(0, 256, m + 1).astype(np.uint8)
        b, eob = _ref(oracle, x[:m])
        for way in ("block-pageable", "block-pinned", "raw-pageable", "raw-pinned", "device-out", "blocks-pinned-out"):
            got, st = _invert(c, way, b, eob)  # (raw: m + 1 rows, the largest raw input)
            assert np.array_equal(got, x[:m]) and st["n_suffixes"] == m + 1, way
        b1, eob1 = _ref(oracle, x)
        LF1 = np.array([eob1], np.uint32)
        for pinned in (False, True):
            big = _host(b1, pinned)
            assert _refused(lambda: c.inverse_block(big[:-1], LF1), big) == -5
            assert _refused(lambda: c.inverse_blocks([big[:-1]], [LF1]), big) == -5
            raw1 = _host(_raw(b1, eob1, 0xEE), pinned)  # m + 2 rows
            assert _refused(lambda: c.inverse_raw(raw1[:-1], LF1), raw1) == -5
        e0 = np.zeros(0, np.uint8)
        assert _refused(lambda: c.inverse_block(e0, np.array([0], np.uint32))) == -1
        one = np.array([0x42, GUARD], np.uint8)
        assert _refused(lambda: c.inverse_raw(one[:1], np.array([0], np.uint32)), one) == -1
        n = 1000
        bb, _ = _ref(oracle, rng.integers(0, 256, n).astype(np.uint8))
        bad = np.array([n + 1], np.uint32)  # eob = N
        for pinned in (False, True):
            h = _host(bb, pinned)
            assert _refused(lambda: c.inverse_block(h[:-1], bad), h) == -1
            assert _refused(lambda: c.inverse_blocks([h[:-1]], [bad]), h) == -1
            assert _refused(lambda: c.inverse_blocks([h[:-1], e0], [[1], [0]]), h) == -1  # an empty block: nothing done
            r = _host(_raw(bb, 5, 0xEE), pinned)
            assert _refused(lambda: c.inverse_raw(r[:-1], bad), r) == -1
        d = _dev(bb)
        dh = d.cpu().numpy()
        assert _refused(lambda: c.inverse_block_device(d.data_ptr(), d.data_ptr(), n, n + 1)) == -1
        assert _refused(lambda: c.inverse_block_device(d.data_ptr(), d.data_ptr(), 0, 0)) == -1
        assert _refused(lambda: c.inverse_block_device(d.data_ptr(), d.data_ptr(), m + 1, 0)) == -5
        torch.cuda.synchronize()
        assert np.array_equal(d.cpu().numpy(), dh), "a refused device call wrote into its buffer"
    finally:
        c.close()


# ---- scratch the inverse shares with the forward transform ------------------------------------------------------------

@pytest.mark.parametrize("knobs", [{}, {"BWTC_LAZY": "2"}, {"BWTC_GRAM": "0"}], ids=["default", "lazy2", "gram0"])
def test_inverse_between_forwards_changes_nothing(oracle, monkeypatch, knobs):
    """The inverse borrows the lazy-rank prefix table (its bucket-start tables), the gram-histogram words (its
    single-cycle check) and d_scat (its splitter arrays): forward(A), inverse(B), forward(A) must give identical bytes,
    LFpowers and freqs, and inverse(B) there must equal inverse(B) on a fresh context."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    a = bw.generate("markov", 3 << 19, seed=900)
    xb = bw.generate("dna", 300001, seed=901)
    bb, eobb = _ref(oracle, xb, 8)
    c = bw.CudaContext(2 << 20)
    fresh = bw.CudaContext(2 << 20)
    try:
        def fwd():
            blk = a.copy()
            LF = np.zeros(8, np.uint32)
            fr = np.zeros(256, np.uint32)
            c.bwt_block(blk, LF, fr)
            return blk, LF, fr

        f1 = fwd()
        got, st = _invert(c, "block-pageable", bb, eobb)
        want, st_fresh = _invert(fresh, "block-pageable", bb, eobb)
        assert np.array_equal(got, xb) and np.array_equal(want, xb)
        assert st["rounds"] == st_fresh["rounds"] and st["kernel_launches"] == st_fresh["kernel_launches"]
        f2 = fwd()
        for u, v, what in zip(f1, f2, ("bytes", "LFpowers", "freqs")):
            assert np.array_equal(u, v), f"forward {what} changed after an inverse on the same context"
        ref_b, ref_lf, ref_fr = oracle.block(a, 8)
        assert np.array_equal(f1[0], ref_b) and np.array_equal(f1[1], ref_lf) and np.array_equal(f1[2], ref_fr)
    finally:
        c.close()
        fresh.close()


def test_short_inverse_after_a_long_one(oracle):
    xl = bw.generate("random", 3 << 20, seed=910)
    bl, eobl = _ref(oracle, xl)
    c = bw.CudaContext(4 << 20)
    fresh = bw.CudaContext(4 << 20)
    try:
        got, _ = _invert(c, "block-pinned", bl, eobl)
        assert np.array_equal(got, xl)
        for n in (1, 5, 31, 33, 1000, 70000):
            xs = bw.generate("markov", n, seed=911 + n)
            bs, eobs = _ref(oracle, xs)
            for way in ("block-pinned", "raw-pageable", "device-out"):
                got, st = _invert(c, way, bs, eobs)
                want, st_fresh = _invert(fresh, way, bs, eobs)
                assert np.array_equal(got, xs) and np.array_equal(want, xs), (n, way)
                assert st["rounds"] == st_fresh["rounds"] == _jump_rounds(n + 1)
            got, _ = _invert(c, "block-pageable", bl, eobl)  # and the long block again
            assert np.array_equal(got, xl)
    finally:
        c.close()
        fresh.close()


# ---- the largest block, checked exactly ---------------------------------------------------------------------------------

def test_maximum_block_round_trip():
    """The 0x7FFFFFFD-byte block of test_maximum_block_size_properties (N = 2^31 - 2 rows): forward, then the in-place
    inverse must return it byte for byte, and so must the same transformed bytes in raw form through inverse_raw.  The
    inverse of a valid input is injective, so this is also an exact check of the forward transform at this size."""
    n = bw.MAX_BLOCK
    try:
        c = bw.CudaContext(n)
    except bw.BwtcCudaError as e:
        pytest.skip(f"cannot allocate scratch for a {n >> 20} MiB block: {e}")
    try:
        x = bw.generate("random", n, seed=33)
        x[12345:12345 + 4096] = x[777:777 + 4096]
        blk = x.copy()
        LF = np.zeros(8, np.uint32)
        c.bwt_block(blk, LF, None)
        eob = int(LF[0])
        raw = np.empty(n + 2, np.uint8)  # N = 2^31 - 2 rows, then a guard byte
        raw[:n] = blk
        raw[n] = blk[eob] if eob < n else 0
        raw[eob] = 0xEE
        raw[n + 1] = GUARD
        last = int(raw[n])
        assert c.inverse_block(blk, LF) == n
        assert c.stats()["n_suffixes"] == n + 1
        assert np.array_equal(blk, x), "the largest block was not restored"
        del blk
        assert c.inverse_raw(raw[:-1], LF) == n
        assert raw[n] == last and raw[n + 1] == GUARD
        assert np.array_equal(raw[:n], x), "the largest block was not restored from its raw form"
    finally:
        c.close()
