"""GPU tests of block integrity: the inverse recognises inputs that are not the BWT of any text (BWTC_CUDA_ECORRUPT,
DESIGN.md §3.7) and the opt-in verification of the forward transform (bwtc_cuda_ctx_set_verify, BWTC_CUDA_EVERIFY,
§3.10).  Mutated oracle outputs are judged by the CPU classifier of tests/test_cabi_verify.py: a valid mutant must restore
to a text whose oracle forward is the mutant, an invalid one must be refused."""
import ctypes

import numpy as np
import pytest

import bwtc_b200 as bw
from test_cabi_verify import classify
from test_gpu_parity import ENGINE_KNOBS, _oracle_generated


def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")]

GUARD = 0x5A
KINDS = ("markov", "dna", "repetitive", "random")
SIZES = (1, 2, 3, 7, 31, 32, 33, 100, 1000, 4096, 65536, 1 << 20)


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(2 << 20)
    yield c
    c.close()


def _mutants(out, eob, rng):
    """Two single-byte changes (to another byte of the block where it has one), two swaps of unequal bytes, two moved
    end-of-block rows: [(label, bytes, eob)]."""
    n = out.size
    res = []
    vals = np.unique(out)
    for _ in range(2):
        m = out.copy()
        i = int(rng.integers(n))
        others = vals[vals != m[i]]
        m[i] = int(rng.choice(others)) if others.size else (int(m[i]) + 1) % 256
        res.append(("byte", m, eob))
    for _ in range(2):
        if vals.size < 2:
            break
        i = int(rng.integers(n))
        js = np.flatnonzero(out != out[i])
        j = int(js[rng.integers(js.size)])
        m = out.copy()
        m[i], m[j] = m[j], m[i]
        res.append(("swap", m, eob))
    for _ in range(2):
        if n == 0:
            break
        e = int(rng.integers(n))
        res.append(("eob", out.copy(), e if e != eob else n))
    return res


def _all_mutants(oracle):
    rng = np.random.default_rng(2024)
    cases = []
    for kind in KINDS:
        for n in SIZES:
            x = bw.generate(kind, n, seed=3000 + n)
            out, LF, _ = oracle.block(x, 8)
            for label, m, e in _mutants(out, int(LF[0]), rng):
                cases.append((kind, n, label, m, e, classify(m, e)))
    return cases


@pytest.fixture(scope="module")
def mutants(oracle):
    cases = _all_mutants(oracle)
    labels = [c[5] for c in cases]
    assert any(v for v, _, _ in labels), "no valid mutant"
    assert any(a for _, a, _ in labels), "no mutant fails test (a)"
    assert any(b for _, _, b in labels), "no mutant fails test (b)"
    assert any(a and not b for _, a, b in labels) and any(b and not a for _, a, b in labels)
    return cases


def _expect_valid(oracle, m, e, restored, what):
    out2, LF2, _ = oracle.block(restored, 1)
    assert np.array_equal(out2, m) and int(LF2[0]) == e, what


def _expect_corrupt(fn, what):
    with pytest.raises(bw.BwtcCudaError) as ei:
        fn()
    assert ei.value.code == bw.ECORRUPT, (what, ei.value)
    assert "not the BWT" in str(ei.value)


def test_inverse_block_detects_corrupt_blocks(ctx, oracle, mutants):
    for kind, n, label, m, e, (valid, _, _) in mutants:
        what = (kind, n, label, e)
        buf = np.append(m, np.uint8(GUARD))
        LF = np.array([e], np.uint32)
        if valid:
            assert ctx.inverse_block(buf[:-1], LF) == n
            _expect_valid(oracle, m, e, buf[:-1].copy(), what)
        else:
            _expect_corrupt(lambda: ctx.inverse_block(buf[:-1], LF), what)
            assert np.array_equal(buf[:-1], m), ("a pageable corrupt block must stay untouched", what)
            assert ctx.stats()["flags"] & bw.FLAG_CORRUPT
        assert buf[-1] == GUARD, what
    ctx.inverse_block(*_valid_pair(oracle))  # the context stays usable


def _valid_pair(oracle):
    x = bw.generate("markov", 5000, seed=9)
    out, LF, _ = oracle.block(x, 8)
    return out, LF


def test_inverse_raw_detects_corrupt_blocks(ctx, oracle, mutants):
    for kind, n, label, m, e, (valid, _, _) in mutants:
        what = (kind, n, label, e)
        raw = np.empty(n + 1, np.uint8)  # raw contract: row N-1 in its own slot, bwt[eob] ignored
        raw[:n] = m
        raw[n] = m[e] if e < n else 0x33
        if e < n:
            raw[e] = 0x77
        LF = np.array([e], np.uint32)
        if valid:
            assert ctx.inverse_raw(raw, LF) == n
            _expect_valid(oracle, m, e, raw[:n].copy(), what)
        else:
            _expect_corrupt(lambda: ctx.inverse_raw(raw, LF), what)


def test_inverse_block_device_detects_corrupt_blocks(ctx, oracle, mutants):
    import torch

    for kind, n, label, m, e, (valid, _, _) in mutants:
        what = (kind, n, label, e)
        d_in = torch.from_numpy(m.copy()).cuda()
        d_out = torch.zeros(n + 1, dtype=torch.uint8, device="cuda")
        d_out[n] = GUARD
        torch.cuda.synchronize()
        if valid:
            assert ctx.inverse_block_device(d_in.data_ptr(), d_out.data_ptr(), n, e) == n
            _expect_valid(oracle, m, e, d_out[:n].cpu().numpy(), what)
        else:
            _expect_corrupt(lambda: ctx.inverse_block_device(d_in.data_ptr(), d_out.data_ptr(), n, e), what)
        assert int(d_out[n]) == GUARD and np.array_equal(d_in.cpu().numpy(), m), what


def _mixed_batch(oracle, rng, count=16, n=20000):
    """count oracle blocks of n bytes (the last shorter) of which about a third are made corrupt (checked with the
    classifier): (texts, transformed bytes, LF rows, corrupt mask)."""
    xs = [bw.generate(KINDS[k % 4], n if k + 1 < count else n // 3, seed=4000 + k) for k in range(count)]
    bwts, LF, bad = [], np.zeros((count, 256), np.uint32), []
    for k, x in enumerate(xs):
        out, lf, _ = oracle.block(x, 8)
        LF[k, : lf.size] = lf
        corrupt = False
        if k % 3 == 1:
            for label, m, e in _mutants(out, int(lf[0]), rng):
                if not classify(m, e)[0]:
                    out, LF[k, 0], corrupt = m, e, True
                    break
        assert classify(out, int(LF[k, 0]))[0] == (not corrupt)
        bwts.append(out)
        bad.append(corrupt)
    assert any(bad) and not all(bad)
    return xs, bwts, LF, bad


@pytest.mark.parametrize("kind", ["pageable", "pinned", "device"])
def test_batch_restores_valid_blocks_and_leaves_corrupt_ones(ctx, oracle, kind):
    import torch

    rng = np.random.default_rng({"pageable": 1, "pinned": 2, "device": 3}[kind])
    xs, bwts, LF, bad = _mixed_batch(oracle, rng)
    count = len(xs)
    if kind == "device":
        bufs = [torch.from_numpy(np.append(b, np.uint8(GUARD))).cuda() for b in bwts]
        blocks = [(t.data_ptr(), t.numel() - 1) for t in bufs]
        torch.cuda.synchronize()
    else:
        bufs = [np.append(b, np.uint8(GUARD)) for b in bwts]
        if kind == "pinned":
            bufs = [torch.from_numpy(b).pin_memory().numpy() for b in bufs]
        blocks = [b[:-1] for b in bufs]
    stats = (bw.Stats * count)()
    rows = np.ascontiguousarray(LF)
    a_in = (ctypes.c_void_p * count)(*[b[0] if kind == "device" else b.ctypes.data for b in blocks])
    sizes = np.array([x.size for x in xs], np.uint32)
    rc = ctx._lib.bwtc_cuda_inverse_blocks(ctx._h, a_in, None, sizes.ctypes.data, count, 1 if kind == "device" else 0,
                                           rows.ctypes.data, ctypes.addressof(stats))
    assert rc == bw.ECORRUPT
    first = bad.index(True)
    assert f"block {first} " in ctx._lib.bwtc_cuda_last_error(ctx._h).decode()
    for k in range(count):
        got = bufs[k].cpu().numpy() if kind == "device" else bufs[k]
        assert got[-1] == GUARD, k
        assert np.array_equal(got[:-1], bwts[k] if bad[k] else xs[k]), (k, bad[k])
        assert bool(stats[k].flags & bw.FLAG_CORRUPT) == bad[k], k
        assert stats[k].batch_blocks == count
        assert (stats[k].flags & ~bw.FLAG_CORRUPT) == (stats[0].flags & ~bw.FLAG_CORRUPT)


@pytest.mark.parametrize("batch", ["1", "0"])
def test_inverse_blocks_binding_reports_corrupt_indices(oracle, monkeypatch, batch):
    """Through CudaContext.inverse_blocks: the batch and the one-by-one path (BWTC_BATCH=0) both restore the valid blocks,
    leave the corrupt ones as they were (pinned buffers too) and name them."""
    import torch

    monkeypatch.setenv("BWTC_BATCH", batch)
    c = bw.CudaContext(2 << 20)
    try:
        rng = np.random.default_rng(5)
        xs, bwts, LF, bad = _mixed_batch(oracle, rng)
        for pinned in (False, True):
            work = [b.copy() for b in bwts]
            if pinned:
                work = [torch.from_numpy(b).pin_memory().numpy() for b in work]
            with pytest.raises(bw.BwtcCudaError) as ei:
                c.inverse_blocks(work, LF)
            assert ei.value.code == bw.ECORRUPT
            assert ei.value.blocks == [k for k in range(len(xs)) if bad[k]]
            assert c.stats()["batch_blocks"] == (len(xs) if batch == "1" else 1)
            for k in range(len(xs)):
                assert np.array_equal(work[k], bwts[k] if bad[k] else xs[k]), (pinned, k)
    finally:
        c.close()


def test_pipeline_fails_only_corrupt_tickets(oracle):
    rng = np.random.default_rng(6)
    n = 1 << 15
    kinds = "FIICIFCIIFIICCIF"  # F forward, I valid inverse, C corrupt inverse
    p = bw.Pipeline(n, depth=2)
    lib = p._lib
    items = []
    try:
        for j, kd in enumerate(kinds):
            x = bw.generate(KINDS[j % 4], n, seed=5000 + j)
            t = ctypes.c_uint64(0)
            if kd == "F":
                blk = x.copy()
                LF = np.zeros(256, np.uint32)
                nLF = ctypes.c_uint32(0)
                rc = lib.bwtc_cuda_pipeline_submit(p._h, blk.ctypes.data, blk.ctypes.data, n, 8, 0, LF.ctypes.data,
                                                   ctypes.addressof(nLF), None, None, ctypes.byref(t))
                items.append((kd, x, blk, LF, nLF, None, t))
            else:
                out, lf, _ = oracle.block(x, 8)
                e = int(lf[0])
                if kd == "C":
                    out, e = next((m, ee) for _, m, ee in _mutants(out, e, rng) if not classify(m, ee)[0])
                blk = out.copy()
                rc = lib.bwtc_cuda_pipeline_submit_inverse(p._h, blk.ctypes.data, blk.ctypes.data, n, e, 0, None,
                                                           ctypes.byref(t))
                items.append((kd, x, blk, None, None, out, t))
            assert rc == 0
        for kd, x, blk, LF, nLF, out, t in reversed(items):
            rc = lib.bwtc_cuda_pipeline_wait(p._h, t.value)
            assert rc == (bw.ECORRUPT if kd == "C" else 0), (kd, t.value, rc)
            if kd == "F":
                b, lf, _ = oracle.block(x, 8)
                assert np.array_equal(blk, b) and np.array_equal(LF[: nLF.value], lf)
            elif kd == "I":
                assert np.array_equal(blk, x)
            else:
                assert np.array_equal(blk, out)
    finally:
        p.close()


def test_pipeline_wait_raises_for_the_corrupt_handle_only(oracle):
    rng = np.random.default_rng(8)
    n = 4096
    xs = [bw.generate("dna", n, seed=5100 + k) for k in range(6)]
    p = bw.Pipeline(n, depth=1)
    try:
        hs, want = [], []
        for k, x in enumerate(xs):
            out, lf, _ = oracle.block(x, 8)
            e = int(lf[0])
            if k == 3:
                out, e = next((m, ee) for _, m, ee in _mutants(out, e, rng) if not classify(m, ee)[0])
            hs.append(p.submit_inverse(out.copy(), [e]))
            want.append(None if k == 3 else x)
        for k, h in enumerate(hs):
            if want[k] is None:
                with pytest.raises(bw.BwtcCudaError) as ei:
                    p.wait(h)
                assert ei.value.code == bw.ECORRUPT
            else:
                assert np.array_equal(p.wait(h), want[k])
    finally:
        p.close()


# ---- forward verification -------------------------------------------------------------------------------------------
def _gpu_block(ctx, x, starts=8):
    blk = np.append(x, np.uint8(0xAB))
    LF = np.zeros(bw.num_starting_points(x.size, starts), np.uint32)
    fr = np.zeros(256, np.uint32)
    ctx.bwt_block(blk[:-1], LF, fr)
    assert blk[-1] == 0xAB
    return blk[:-1].copy(), LF, fr


@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()) or "default")
def test_verified_forward_is_bit_exact_under_every_engine_path(oracle, monkeypatch, knobs):
    """The blocks and batches of test_gpu_parity.py::test_every_engine_path_is_bit_exact with verification on: same bytes,
    LFpowers and freqs as the oracle (and so as verification off), stats bit 6 set; with verification off it is clear."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    n = (2 << 20) + 4097
    ctx = bw.CudaContext(n)
    rng = np.random.default_rng(77)
    cases = [("markov", n), ("dna", n), ("repetitive", 1 << 20), ("repetitive", n - 5), ("random", n - 4099)]
    try:
        ctx.set_verify(True)
        for kind, sz in cases:
            x = bw.generate(kind, sz, seed=41)
            if kind == "random":
                x[rng.integers(0, sz, 1000)] = 0
            want = _oracle_generated(oracle, kind + "+zeros" if kind == "random" else kind, 41, sz, x)
            got = _gpu_block(ctx, x)
            for g, w in zip(got, want):
                assert np.array_equal(g, w), (kind, knobs)
            assert ctx.stats()["flags"] & bw.FLAG_VERIFIED, kind
        for kind, sizes in (("markov", [1 << 18] * 8 + [4000]), ("dna", [1 << 18] * 8 + [4000]), ("repetitive", [1 << 18] * 4)):
            xs = [np.minimum(bw.generate(kind, sz, seed=60 + k), 254) for k, sz in enumerate(sizes)]
            bufs = [np.append(x, np.uint8(0xAB)) for x in xs]
            LF, nLF, fr = ctx.bwt_blocks([b[:-1] for b in bufs], 8)
            st = ctx.stats()
            assert st["flags"] & 2 and st["flags"] & bw.FLAG_VERIFIED and st["batch_blocks"] == len(xs), (kind, st["flags"])
            for k, x in enumerate(xs):
                want = _oracle_generated(oracle, kind, 60 + k, x.size, x)
                assert bufs[k][-1] == 0xAB
                assert np.array_equal(bufs[k][:-1], want[0]), (kind, k, knobs)
                assert nLF[k] == want[1].size and np.array_equal(LF[k, : nLF[k]], want[1]), (kind, k, knobs)
                assert np.array_equal(fr[k], want[2]), (kind, k, knobs)
        ctx.set_verify(False)
        x = bw.generate("markov", n, seed=41)
        got = _gpu_block(ctx, x)
        assert np.array_equal(got[0], _oracle_generated(oracle, "markov", 41, n, x)[0])
        assert not ctx.stats()["flags"] & bw.FLAG_VERIFIED
    finally:
        ctx.close()


def test_verify_off_runs_the_same_kernels(oracle):
    """Verification off is the engine as it was: the same launch count with the switch never touched and switched off;
    on, the inverse and the comparison come on top."""
    x = bw.generate("markov", 1 << 20, seed=12)
    a, b = bw.CudaContext(1 << 20), bw.CudaContext(1 << 20)
    try:
        b.set_verify(True)
        b.set_verify(False)
        ra, rb = _gpu_block(a, x), _gpu_block(b, x)
        la, lb = a.stats()["kernel_launches"], b.stats()["kernel_launches"]
        assert la == lb and all(np.array_equal(u, v) for u, v in zip(ra, rb))
        b.set_verify(True)
        rc = _gpu_block(b, x)
        assert all(np.array_equal(u, v) for u, v in zip(ra, rc))
        assert b.stats()["kernel_launches"] > la
    finally:
        a.close()
        b.close()


def _expect_everify(fn):
    with pytest.raises(bw.BwtcCudaError) as ei:
        fn()
    assert ei.value.code == bw.EVERIFY, ei.value


def test_corrupted_output_gives_everify_and_keeps_inputs(oracle, monkeypatch):
    import torch

    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_OUT", "1")
    n = 100000
    ctx = bw.CudaContext(16 * (n + 1))
    monkeypatch.delenv("BWTC_DEBUG_CORRUPT_OUT")
    good = bw.CudaContext(16 * (n + 1))
    try:
        ctx.set_verify(True)
        good.set_verify(True)
        x = bw.generate("markov", n, seed=13)
        want = oracle.block(x, 8)
        for kind in ("pageable", "pinned"):
            buf = np.append(x, np.uint8(GUARD))
            if kind == "pinned":
                buf = torch.from_numpy(buf).pin_memory().numpy()
            LF = np.full(8, 0xDEAD, np.uint32)
            fr = np.full(256, 3, np.uint32)
            _expect_everify(lambda: ctx.bwt_block(buf[:-1], LF, fr))
            assert np.array_equal(buf[:-1], x) and buf[-1] == GUARD, kind
            assert (LF == 0xDEAD).all() and (fr == 3).all(), kind
            assert ctx.stats()["flags"] & bw.FLAG_VERIFIED
            assert "does not restore" in ctx._lib.bwtc_cuda_last_error(ctx._h).decode()
        d = torch.from_numpy(np.append(x, np.uint8(GUARD))).cuda()
        torch.cuda.synchronize()
        LF = np.zeros(8, np.uint32)
        _expect_everify(lambda: ctx.bwt_block_device(d.data_ptr(), d.data_ptr(), n, LF, None))
        assert np.array_equal(d.cpu().numpy(), np.append(x, np.uint8(GUARD))), "in-place device block must be rewritten"
        xs = [bw.generate("dna", n, seed=14 + k) for k in range(6)]
        for on_device in (False, True):
            if on_device:
                ts = [torch.from_numpy(v.copy()).cuda() for v in xs]
                torch.cuda.synchronize()
                _expect_everify(lambda: ctx.bwt_blocks(ts, 8, on_device=True))
                assert all(np.array_equal(t.cpu().numpy(), v) for t, v in zip(ts, xs))
            else:
                bs = [v.copy() for v in xs]
                _expect_everify(lambda: ctx.bwt_blocks(bs, 8))
                assert all(np.array_equal(b, v) for b, v in zip(bs, xs))
            assert ctx.stats()["batch_blocks"] == 6 and ctx.stats()["flags"] & bw.FLAG_VERIFIED
        # the context stays usable: verification off, the same context transforms correctly
        ctx.set_verify(False)
        got = _gpu_block(ctx, x)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        got = _gpu_block(good, x)  # and a context without the hook passes verification
        assert np.array_equal(got[0], want[0]) and good.stats()["flags"] & bw.FLAG_VERIFIED
    finally:
        ctx.close()
        good.close()


def test_corrupted_output_fails_its_pipeline_ticket(monkeypatch):
    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_OUT", "1")
    p = bw.Pipeline(1 << 16, depth=1)
    monkeypatch.delenv("BWTC_DEBUG_CORRUPT_OUT")
    try:
        p.set_verify(True)
        x = bw.generate("markov", 50000, seed=15)
        blk = x.copy()
        h = p.submit(blk, 8)
        with pytest.raises(bw.BwtcCudaError) as ei:
            p.wait(h)
        assert ei.value.code == bw.EVERIFY
        assert np.array_equal(blk, x)
    finally:
        p.close()


def test_pipeline_verified_round_trip(oracle):
    xs = [bw.generate(KINDS[k % 4], 30000 if k % 5 else 7777, seed=5200 + k) for k in range(24)]
    blocks = [x.copy() for x in xs]
    p = bw.Pipeline(1 << 15, depth=3)
    try:
        p.set_verify(True)
        LF, nLF, _, stats = p.run(blocks, 8)
        assert all(s["flags"] & bw.FLAG_VERIFIED for s in stats)
        for k, x in enumerate(xs):
            b, lf, _ = oracle.block(x, 8)
            assert np.array_equal(blocks[k], b) and np.array_equal(LF[k, : nLF[k]], lf), k
    finally:
        p.close()


def test_verified_32mib_markov_block(oracle_record):
    n = 32 << 20
    x = bw.generate("markov", n, seed=31)
    ctx = bw.CudaContext(n)
    try:
        ctx.set_verify(True)
        out = x.copy()
        LF = np.zeros(8, np.uint32)
        fr = np.zeros(256, np.uint32)
        ctx.bwt_block(out, LF, fr)
        st = ctx.stats()
    finally:
        ctx.close()
    assert st["flags"] & bw.FLAG_VERIFIED
    oracle_record.check(x, 8, out, LF, fr)
    print(f"verified forward 32 MiB markov: gpu_ms={st['gpu_ms']:.3f}, {st['kernel_launches']} launches")
