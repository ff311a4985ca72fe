"""GPU tests of the BATCHED inverse transform (bwtc_cuda_inverse_blocks, bwtc_cuda_pipeline_submit_inverse; DESIGN.md §3.7):
equal-sized blocks inverted as one device-side problem.  Every block's expected bytes come from the oracle (its forward
transform, then its inverse), every block carries a guard byte after it that must survive, and batched results must equal
the single-block path byte for byte."""
import ctypes
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
KINDS = ("markov", "dna", "repetitive", "random")


def _guarded(arrays):
    """Copies of the arrays, each a view into a buffer with one guard byte behind it."""
    bufs = []
    for a in arrays:
        b = np.empty(a.size + 1, np.uint8)
        b[:-1] = a
        b[-1] = GUARD
        bufs.append(b)
    return bufs, [b[:-1] for b in bufs]


def _forward(oracle, xs, starts):
    """Oracle forward transform of every block: (transformed bytes, LFpowers rows [count, 256]); the oracle's own inverse
    is checked to restore each block."""
    bwts, LF = [], np.zeros((len(xs), 256), np.uint32)
    for k, x in enumerate(xs):
        b, lf, _ = oracle.block(x, starts)
        assert np.array_equal(oracle.inverse_block(b, lf[0]), x)
        bwts.append(b)
        LF[k, : lf.size] = lf
    return bwts, LF


def _check_inverse(ctx, oracle, xs, starts=8):
    """inverse_blocks on guarded copies of the oracle's forward output: every block restored, guards intact."""
    bwts, LF = _forward(oracle, xs, starts)
    bufs, views = _guarded(bwts)
    ctx.inverse_blocks(views, LF)
    for k, (b, x) in enumerate(zip(bufs, xs)):
        assert b[-1] == GUARD, f"byte after block {k} was written"
        assert np.array_equal(b[:-1], x), f"block {k} of {len(xs)} (n={x.size}) not restored"
    return ctx.stats()


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(8 << 20)
    yield c
    c.close()


def test_batch_forms_and_restores_markov_blocks(ctx, oracle):
    xs = [bw.generate("markov", 1 << 18, seed=500 + k) for k in range(15)] + [bw.generate("markov", 77777, seed=499)]
    for starts in (1, 8):
        st = _check_inverse(ctx, oracle, xs, starts)
        assert st["n_suffixes"] == sum(x.size + 1 for x in xs), "the 16 blocks must have been inverted as one batch"
        assert st["batch_blocks"] == 16 and st["flags"] & 2


@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 255, 256, 257])
def test_tiny_blocks_batch_and_split_into_runs(ctx, oracle, n):
    rng = np.random.default_rng(n)
    xs = [rng.integers(0, (2, 4, 256)[k % 3], n).astype(np.uint8) for k in range(64)]
    st = _check_inverse(ctx, oracle, xs)
    assert st["batch_blocks"] == 64 and st["n_suffixes"] == 64 * (n + 1)
    st = _check_inverse(ctx, oracle, xs + [xs[5].copy()])  # 65 blocks: a run of 64, then one on its own
    assert st["batch_blocks"] == 1 and st["n_suffixes"] == n + 1


def test_row_stride_multiple_of_32_and_not(ctx, oracle):
    rng = np.random.default_rng(3)
    for n0, nl in ((1023, 1023), (1023, 500), (1024, 1024), (2047, 31), (4095, 4064), (3000, 1)):
        xs = [rng.integers(0, 7, n0).astype(np.uint8) for _ in range(5)] + [rng.integers(0, 7, nl).astype(np.uint8)]
        st = _check_inverse(ctx, oracle, xs)
        assert st["batch_blocks"] == 6


def test_degenerate_blocks(ctx, oracle):
    """All-equal blocks (end-of-block row N-1), blocks of 0x00 bytes, two-letter blocks."""
    rng = np.random.default_rng(4)
    same = [np.full(4000, v, np.uint8) for v in (0x00, 0x41, 0xFF, 0x00, 0x7F)]
    bwts, LF = _forward(oracle, same, 8)
    assert any(int(LF[k, 0]) == 4000 for k in range(len(same))), "expected an end-of-block row at N - 1"
    st = _check_inverse(ctx, oracle, same)
    assert st["batch_blocks"] == 5
    zeros = [np.zeros(9000, np.uint8) for _ in range(3)] + [np.zeros(100, np.uint8)]
    assert _check_inverse(ctx, oracle, zeros)["batch_blocks"] == 4
    two = [rng.integers(0, 2, 20000).astype(np.uint8) * 0xFF for _ in range(4)]
    two += [np.frombuffer(b"ab" * 10000, np.uint8).copy()]
    assert _check_inverse(ctx, oracle, two)["batch_blocks"] == 5


def test_all_256_byte_values_still_batch(ctx, oracle):
    """Unlike the forward batch, the inverse reserves no byte value: blocks using all 256 values are batched."""
    rng = np.random.default_rng(5)
    xs = []
    for k in range(6):
        x = rng.integers(0, 256, 30000).astype(np.uint8)
        x[rng.choice(30000, 256, replace=False)] = rng.permutation(256).astype(np.uint8)
        xs.append(x)
    xs[-1] = xs[-1][:12345].copy()
    xs[-1][:256] = np.arange(256, dtype=np.uint8)
    assert all(np.unique(x).size == 256 for x in xs)
    st = _check_inverse(ctx, oracle, xs)
    assert st["n_suffixes"] == sum(x.size + 1 for x in xs) and st["flags"] & 2


def test_repetitive_and_unequal_sizes(ctx, oracle):
    rep = [bw.generate("repetitive", 1 << 17, seed=7 + k) for k in range(4)]
    assert _check_inverse(ctx, oracle, rep)["batch_blocks"] == 4
    mixed = [bw.generate("dna", n, seed=n) for n in (40000, 40000, 40000, 1000, 50000, 50000, 1, 2, 2)]
    _check_inverse(ctx, oracle, mixed, 256)


def test_batch_equals_single_and_unbatched_context(ctx, oracle, monkeypatch):
    rng = np.random.default_rng(6)
    xs = [bw.generate(KINDS[k % 4], 70000, seed=600 + k) for k in range(9)] + [rng.integers(0, 256, 7).astype(np.uint8)]
    xs += [bw.generate("markov", 3000, seed=k) for k in range(5)]
    bwts, LF = _forward(oracle, xs, 8)
    batched = [b.copy() for b in bwts]
    ctx.inverse_blocks(batched, LF)
    single = [b.copy() for b in bwts]
    for k, b in enumerate(single):
        ctx.inverse_block(b, LF[k, :1].copy())
    monkeypatch.setenv("BWTC_BATCH", "0")
    c0 = bw.CudaContext(8 << 20)
    try:
        unbatched = [b.copy() for b in bwts]
        c0.inverse_blocks(unbatched, LF)
        assert c0.stats()["batch_blocks"] == 1
    finally:
        c0.close()
    for k, x in enumerate(xs):
        assert np.array_equal(batched[k], single[k]) and np.array_equal(batched[k], unbatched[k]), k
        assert np.array_equal(batched[k], x), k


def test_buffer_kinds(ctx, oracle):
    import torch

    xs = [bw.generate("markov", 50000, seed=700 + k) for k in range(7)] + [bw.generate("markov", 20000, seed=699)]
    bwts, LF = _forward(oracle, xs, 8)
    # pinned, in place
    pinned = [torch.from_numpy(b.copy()).pin_memory() for b in bwts]
    ctx.inverse_blocks([t.numpy() for t in pinned], LF)
    assert ctx.stats()["batch_blocks"] == 8
    for t, x in zip(pinned, xs):
        assert np.array_equal(t.numpy(), x)
    # separate outputs (guarded); the inputs stay as they were
    src = [b.copy() for b in bwts]
    obufs, outs = _guarded([np.zeros_like(b) for b in bwts])
    ctx.inverse_blocks(src, LF, out=outs)
    for k, x in enumerate(xs):
        assert np.array_equal(src[k], bwts[k]) and obufs[k][-1] == GUARD and np.array_equal(outs[k], x)
    # device tensors, in place and into separate device outputs
    dev = [torch.from_numpy(b.copy()).cuda() for b in bwts]
    dout = [torch.zeros_like(t) for t in dev]
    ctx.inverse_blocks(dev, LF, on_device=True, out=dout)
    ctx.inverse_blocks(dev, LF, on_device=True)
    torch.cuda.synchronize()
    for t, o, x in zip(dev, dout, xs):
        assert np.array_equal(t.cpu().numpy(), x) and np.array_equal(o.cpu().numpy(), x)


def test_forward_then_inverse_on_the_same_device_tensors(ctx):
    import torch

    xs = [bw.generate(KINDS[k % 4], 1 << 16, seed=800 + k) for k in range(12)] + [bw.generate("dna", 999, seed=1)]
    dev = [torch.from_numpy(x.copy()).cuda() for x in xs]
    LF, nLF, _ = ctx.bwt_blocks(dev, 8, want_freqs=False, on_device=True)
    torch.cuda.synchronize()
    assert not np.array_equal(dev[0].cpu().numpy(), xs[0])
    ctx.inverse_blocks(dev, LF, on_device=True)
    torch.cuda.synchronize()
    assert ctx.stats()["batch_blocks"] == len(xs)
    for t, x in zip(dev, xs):
        assert np.array_equal(t.cpu().numpy(), x)


def test_watchdog_retry_restores_pinned_in_place_blocks(oracle, monkeypatch):
    import torch

    monkeypatch.setenv("BWTC_DEBUG_FAKE_WATCHDOG", "1")
    c = bw.CudaContext(4 << 20)
    try:
        xs = [bw.generate("markov", 1 << 17, seed=900 + k) for k in range(6)] + [bw.generate("random", 5000, seed=9)]
        bwts, LF = _forward(oracle, xs, 8)
        pinned = [torch.from_numpy(b.copy()).pin_memory() for b in bwts]
        c.inverse_blocks([t.numpy() for t in pinned], LF)
        st = c.stats()
    finally:
        c.close()
    assert st["flags"] & 1, "the retry with ticket tile ids must have run"
    assert st["flags"] & 2 and st["batch_blocks"] == 7
    for t, x in zip(pinned, xs):
        assert np.array_equal(t.numpy(), x)


def test_pipeline_submit_inverse_waited_in_reverse(oracle):
    xs = [bw.generate(KINDS[k % 4], 1 << 16, seed=1000 + k) for k in range(37)] + [bw.generate("markov", 12345, seed=3)]
    bwts, LF = _forward(oracle, xs, 8)
    bufs, views = _guarded(bwts)
    p = bw.Pipeline(1 << 16, depth=3)
    try:
        handles = [p.submit_inverse(v, LF[k]) for k, v in enumerate(views)]
        for h in reversed(handles):
            p.wait(h)
    finally:
        p.close()
    for b, x in zip(bufs, xs):
        assert b[-1] == GUARD and np.array_equal(b[:-1], x)


def test_pipeline_mixed_forward_and_inverse_stream(oracle):
    """Forward and inverse items interleaved on one pipeline: each is right, and no batch mixes the two kinds."""
    rng = np.random.default_rng(11)
    n = 1 << 15
    kinds = "FFIIIFIFFFIIIIIFIFI"
    fwd_x = [bw.generate("markov", n, seed=1100 + k) for k in range(kinds.count("F"))]
    inv_x = [bw.generate("dna", n, seed=1200 + k) for k in range(kinds.count("I"))]
    inv_bwt, inv_LF = _forward(oracle, inv_x, 8)
    p = bw.Pipeline(n, depth=2)
    lib = p._lib
    items = []
    fi = ii = 0
    try:
        for kd in kinds:
            st = bw.Stats()
            t = ctypes.c_uint64(0)
            if kd == "F":
                blk = fwd_x[fi].copy()
                LF = np.zeros(256, np.uint32)
                nLF = ctypes.c_uint32(0)
                rc = lib.bwtc_cuda_pipeline_submit(p._h, blk.ctypes.data, blk.ctypes.data, n, 8, 0, LF.ctypes.data,
                                                   ctypes.addressof(nLF), None, ctypes.byref(st), ctypes.byref(t))
                items.append(("F", fi, blk, LF, nLF, st, t))
                fi += 1
            else:
                blk = inv_bwt[ii].copy()
                rc = lib.bwtc_cuda_pipeline_submit_inverse(p._h, blk.ctypes.data, blk.ctypes.data, n, int(inv_LF[ii, 0]), 0,
                                                           ctypes.byref(st), ctypes.byref(t))
                items.append(("I", ii, blk, None, None, st, t))
                ii += 1
            assert rc == 0
        tickets = [it[6].value for it in items]
        assert tickets == sorted(tickets) and len(set(tickets)) == len(tickets), "one ticket sequence for both kinds"
        for it in rng.permutation(len(items)):
            assert lib.bwtc_cuda_pipeline_wait(p._h, items[it][6].value) == 0
    finally:
        p.close()
    for kd, idx, blk, LF, nLF, st, _ in items:
        if kd == "F":
            b, lf, _ = oracle.block(fwd_x[idx], 8)
            assert np.array_equal(blk, b) and np.array_equal(LF[: nLF.value], lf)
        else:
            assert np.array_equal(blk, inv_x[idx])
    # a batch holds only consecutive items of one kind: no item's batch is larger than the run of its kind it sits in
    pos = 0
    for _, grp in itertools.groupby(kinds):
        r = len(list(grp))
        for j in range(r):
            assert items[pos + j][5].batch_blocks <= r, (pos + j, kinds)
        pos += r


def test_pipeline_forward_then_inverse_round_trip():
    rng = np.random.default_rng(12)
    for trial in range(3):
        sizes = rng.choice([1, 100, 4096, 60000, 1 << 16], size=40)
        xs = [bw.generate(KINDS[int(rng.integers(0, 4))], int(s), seed=int(rng.integers(1, 1 << 30))) for s in sizes]
        blocks = [x.copy() for x in xs]
        p = bw.Pipeline(1 << 16, depth=3)
        try:
            LF, nLF, freqs, stats = p.run(blocks, 8)
            p.run_inverse(blocks, LF)
        finally:
            p.close()
        for b, x in zip(blocks, xs):
            assert np.array_equal(b, x), trial


def test_argument_errors_leave_every_buffer_untouched(ctx, oracle):
    xs = [bw.generate("markov", 4000, seed=1300 + k) for k in range(5)]
    bwts, LF = _forward(oracle, xs, 8)

    def expect(code, blocks, lf, **kw):
        before = [b.copy() for b in blocks if isinstance(b, np.ndarray)]
        with pytest.raises(bw.BwtcCudaError) as ei:
            ctx.inverse_blocks(blocks, lf, **kw)
        assert ei.value.code == code, ei.value
        for b, c in zip([b for b in blocks if isinstance(b, np.ndarray)], before):
            assert np.array_equal(b, c)

    bad = LF.copy()
    bad[3, 0] = 4001  # end-of-block row outside [0, N) in one block of a batch
    expect(-1, [b.copy() for b in bwts], bad)
    big = np.zeros((8 << 20) + 1, np.uint8)  # above the context capacity
    expect(-5, [b.copy() for b in bwts[:2]] + [big] + [b.copy() for b in bwts[2:]],
           np.concatenate([LF[:2], np.zeros((1, 256), np.uint32), LF[2:]]))
    expect(-1, [b.copy() for b in bwts[:3]] + [(0, 4000)] + [bwts[4].copy()], LF)     # null pointer
    expect(-1, [b.copy() for b in bwts[:3]] + [np.zeros(0, np.uint8)] + [bwts[4].copy()], LF)  # empty block


@pytest.mark.parametrize("kind,count", [("markov", 32), ("random", 16)])
def test_full_size_forward_then_inverse(oracle, kind, count):
    n = 1 << 20
    xs = [bw.generate(kind, n, seed=1400 + k) for k in range(count)]
    c = bw.CudaContext(count * (n + 1))
    try:
        blocks = [x.copy() for x in xs]
        LF, nLF, _ = c.bwt_blocks(blocks, 8)
        for k in range(count):
            b, lf, _ = oracle.block(xs[k], 8)
            assert np.array_equal(blocks[k], b) and np.array_equal(LF[k, : nLF[k]], lf), k
        c.inverse_blocks(blocks, LF)
        st = c.stats()
    finally:
        c.close()
    assert st["batch_blocks"] == count and st["n_suffixes"] == count * (n + 1)
    for b, x in zip(blocks, xs):
        assert np.array_equal(b, x)
    print(f"inverse batch {count} x 1 MiB {kind}: gpu_ms={st['gpu_ms']:.3f}, {st['kernel_launches']} launches")
