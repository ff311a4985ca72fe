"""GPU tests of the verified raw contract and of the LFpowers check (DESIGN.md §3.10): with verification on, a raw
bwtc_cuda_divbwt / divbwtf call is inverted on the device with the text's own last byte as the key of its end-of-text row,
every LFpowers entry (raw, single block, batch, pipeline) is checked against the row the device-side walk visits at its
text position, and BWTC_VERIFY=1 switches verification on for every context created afterwards."""
import numpy as np
import pytest

import bwtc_b200 as bw
from test_gpu_parity import ENGINE_KNOBS
from test_gpu_raw_contract import (F_LAZY, F_TICKETS, GUARD, KINDS, LAST_BYTE_FORMS, N_ENGINE, assert_raw, engine_cases,
                                   last_byte_form, raw_from_block, raw_text, run_raw)


def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")]


def _verified(ctx):
    return bool(ctx.stats()["flags"] & bw.FLAG_VERIFIED)


def _expect_everify(fn, what=None):
    with pytest.raises(bw.BwtcCudaError) as ei:
        fn()
    assert ei.value.code == bw.EVERIFY, (what, ei.value)


def _pinned_copy(a):
    import torch

    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t, t.numpy()


# ---- bit-exact with verification on --------------------------------------------------------------------------------
@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()) or "default")
def test_verified_raw_is_bit_exact_under_every_engine_path(oracle, monkeypatch, knobs):
    """The raw texts of test_every_engine_path_raw (four families x five last-byte forms, about 2 MiB) with verification
    on: U, pidx, LFpowers and freqs equal the oracle's, and every call is marked verified."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    tickets = knobs.get("BWTC_STATIC_TILES") == "0" or knobs.get("BWTC_DEBUG_FAKE_WATCHDOG") == "1"
    ctx = bw.CudaContext(N_ENGINE)
    try:
        ctx.set_verify(True)
        for name, T, want in engine_cases(oracle):
            assert_raw(run_raw(ctx, T, 8), want, (name, knobs))
            st = ctx.stats()
            assert st["flags"] & bw.FLAG_VERIFIED, (name, st["flags"])
            assert bool(st["flags"] & F_TICKETS) == tickets, (name, st["flags"])
            if knobs.get("BWTC_LAZY") == "2":
                assert st["flags"] & F_LAZY, name
    finally:
        ctx.close()


@pytest.fixture(scope="module")
def vctx():
    c = bw.CudaContext(1 << 20)
    c.set_verify(True)
    yield c
    c.close()


def test_verified_raw_last_byte_forms_and_small_texts(oracle, vctx):
    """Every last-byte form on 100 KB texts of the four families; every 2-byte text over {0, 1, 7, 255}; texts whose
    pidx is N - 1; the one-LFpower-per-suffix case (N / nLF = 1, T[N-2] < T[N-1]), whose LFpowers[1] is the row of the
    end-of-text suffix itself."""
    rng = np.random.default_rng(700)
    for kind in KINDS:
        for form in LAST_BYTE_FORMS:
            R = np.ascontiguousarray(bw.generate(kind, 99999, seed=44)[::-1])
            T = last_byte_form(R, form, rng)
            assert_raw(run_raw(vctx, T, 8), oracle.raw(T, 8), (kind, form))
            assert _verified(vctx), (kind, form)
    for a in (0, 1, 7, 255):
        for b in (0, 1, 7, 255):
            T = np.array([a, b], np.uint8)
            for nLF in (1, 2):
                assert_raw(run_raw(vctx, T, nLF), oracle.raw(T, nLF), (a, b, nLF))
                assert _verified(vctx)
    for n in (3, 33, 5000):
        T = np.append(np.uint8(200), rng.integers(0, 200, n - 1).astype(np.uint8))  # suffix 0 is the largest
        want = oracle.raw(T, 8 if n > 8 else n)
        assert want[0] == n - 1
        assert_raw(run_raw(vctx, T, want[2].size), want, ("pidx = N-1", n))
    quirks = 0
    for N, nLF in ((256, 256), (257, 256), (2, 2), (3, 3)):
        for sigma in (2, 4, 256):
            T = rng.integers(0, sigma, N).astype(np.uint8)
            if T[-2] == T[-1]:
                T[-1] ^= 1
            if T[-2] > T[-1]:
                T[-2], T[-1] = T[-1], T[-2]
            assert_raw(run_raw(vctx, T, nLF), oracle.raw(T, nLF), ("quirk", N, sigma))
            assert _verified(vctx)
            quirks += 1
    assert quirks == 12


@pytest.mark.parametrize("m", [1, 4096, 100000])
def test_verified_raw_at_capacity_plus_one(oracle, m):
    rng = np.random.default_rng(710 + m)
    c = bw.CudaContext(m)
    try:
        c.set_verify(True)
        T = np.append(rng.integers(0, 4, m), 2).astype(np.uint8)  # m + 1 bytes, last byte inside the alphabet
        nLF = min(T.size, 8)
        assert_raw(run_raw(c, T, nLF), oracle.raw(T, nLF), m)
        assert _verified(c)
    finally:
        c.close()


def test_verified_raw_buffer_kinds(oracle, vctx):
    """Pageable and pinned buffers, in place (T == U) and into a separate U prefilled with a marker, which U[pidx] keeps."""
    rng = np.random.default_rng(720)
    T = np.append(rng.integers(0, 64, 300000), 17).astype(np.uint8)
    rc, wU, wLF, wfr = oracle.raw(T, 8)
    keep = np.arange(T.size) != rc
    hold = []
    for pinned in (False, True):
        for separate in (False, True):
            tbuf = np.append(T, np.uint8(GUARD))
            ubuf = np.full(T.size + 1, 0xEE, np.uint8)
            ubuf[-1] = GUARD
            if pinned:
                (tt, tbuf), (tu, ubuf) = _pinned_copy(tbuf), _pinned_copy(ubuf)
                hold += [tt, tu]
            src = tbuf[:-1]
            U = ubuf[:-1] if separate else src
            LF = np.zeros(8, np.uint32)
            fr = np.zeros(256, np.uint32)
            what = (pinned, separate)
            assert vctx.divbwtf(src, U, LF, fr) == rc, what
            assert _verified(vctx), what
            assert tbuf[-1] == GUARD and ubuf[-1] == GUARD, what
            assert np.array_equal(LF, wLF) and np.array_equal(fr, wfr), what
            assert np.array_equal(U[keep], wU[keep]), what
            assert U[rc] == (0xEE if separate else T[rc]), what
            if separate:
                assert np.array_equal(src, T), what


def test_verified_raw_32mib_markov(oracle_record):
    """T = reverse(X)·0x00 of the 32 MiB Markov block: the verified block result matches the recorded oracle digests, the
    verified raw result is exactly the one derived from it."""
    x = bw.generate("markov", 32 << 20, seed=31)
    n = x.size
    ctx = bw.CudaContext(n + 1)
    try:
        ctx.set_verify(True)
        blk = x.copy()
        LF = np.zeros(8, np.uint32)
        fr = np.zeros(256, np.uint32)
        p = ctx.bwt_block(blk, LF, fr)
        assert _verified(ctx)
        oracle_record.check(x, 8, blk, LF, fr)
        T = raw_text(x)
        got = run_raw(ctx, T, 8)
        st = ctx.stats()
    finally:
        ctx.close()
    assert st["flags"] & bw.FLAG_VERIFIED
    assert_raw(got, (p, raw_from_block(T, blk, p), LF, fr), "32 MiB markov raw")
    print(f"verified raw 32 MiB markov: gpu_ms={st['gpu_ms']:.3f}, {st['kernel_launches']} launches")


# ---- corruption is found ---------------------------------------------------------------------------------------------
def test_corrupted_raw_output_gives_everify_and_keeps_buffers(oracle, monkeypatch):
    """BWTC_DEBUG_CORRUPT_OUT=1 on raw calls (the flipped row is never pidx, also when pidx is the row the hook picks first):
    EVERIFY, and U (in place or separate), LFpowers and freqs hold what they held before, pageable and pinned; the context
    then transforms correctly with verification off."""
    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_OUT", "1")
    N = 200001
    ctx = bw.CudaContext(N)
    monkeypatch.delenv("BWTC_DEBUG_CORRUPT_OUT")
    rng = np.random.default_rng(730)
    try:
        ctx.set_verify(True)
        half = N // 2  # T[0] = 0x80, unique, with exactly N / 2 smaller bytes: pidx = N / 2
        rest = np.concatenate([rng.integers(0, 0x80, half), rng.integers(0x81, 0x100, N - 1 - half)]).astype(np.uint8)
        rng.shuffle(rest)
        texts = [np.append(np.uint8(0x80), rest), np.append(rng.integers(0, 4, N - 1), 3).astype(np.uint8)]
        assert oracle.raw(texts[0], 8)[0] == half
        hold = []
        for T in texts:
            for pinned in (False, True):
                for separate in (False, True):
                    tbuf = np.append(T, np.uint8(GUARD))
                    ubuf = np.full(N + 1, 0xEE, np.uint8)
                    if pinned:
                        (tt, tbuf), (tu, ubuf) = _pinned_copy(tbuf), _pinned_copy(ubuf)
                        hold += [tt, tu]
                    src = tbuf[:-1]
                    U = ubuf[:-1] if separate else src
                    LF = np.full(8, 0xDEAD, np.uint32)
                    fr = np.full(256, 3, np.uint32)
                    what = (int(T[0]), pinned, separate)
                    _expect_everify(lambda: ctx.divbwtf(src, U, LF, fr), what)
                    assert np.array_equal(src, T) and tbuf[-1] == GUARD, what
                    if separate:
                        assert (ubuf == 0xEE).all(), what
                    assert (LF == 0xDEAD).all() and (fr == 3).all(), what
                    assert _verified(ctx), what
                    assert "does not restore" in ctx._lib.bwtc_cuda_last_error(ctx._h).decode()
        ctx.set_verify(False)
        for T in texts:
            assert_raw(run_raw(ctx, T, 8), oracle.raw(T, 8), "after EVERIFY")
    finally:
        ctx.close()


@pytest.mark.parametrize("j", [1, 4, 7])
def test_wrong_starting_point_is_found(oracle, monkeypatch, j):
    """BWTC_DEBUG_CORRUPT_LF=j changes the device's LFpowers[j] (of every block that has one) before the check: a single
    block, a batch and a raw call with 8 starting points return EVERIFY and leave LFpowers and freqs as they were; calls
    with at most j starting points are unaffected.  On a pipeline only the ticket with 8 starting points fails."""
    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_LF", str(j))
    n = 100000
    ctx = bw.CudaContext(8 * (n + 1))
    p = bw.Pipeline(n, depth=1)
    monkeypatch.delenv("BWTC_DEBUG_CORRUPT_LF")
    try:
        ctx.set_verify(True)
        p.set_verify(True)
        x = bw.generate("markov", n, seed=740)
        blk = x.copy()
        LF = np.full(8, 0xDEAD, np.uint32)
        fr = np.full(256, 3, np.uint32)
        _expect_everify(lambda: ctx.bwt_block(blk, LF, fr), "block")
        assert np.array_equal(blk, x) and (LF == 0xDEAD).all() and (fr == 3).all()
        assert "block 0 of 1" in ctx._lib.bwtc_cuda_last_error(ctx._h).decode()
        LFj = np.zeros(j, np.uint32)
        ctx.bwt_block(blk, LFj, None)  # j starting points: LFpowers[j] does not exist
        assert _verified(ctx) and np.array_equal(blk, oracle.block(x, j)[0])
        xs = [bw.generate("dna", n, seed=741 + k) for k in range(6)]
        bs = [v.copy() for v in xs]
        _expect_everify(lambda: ctx.bwt_blocks(bs, 8), "batch")
        assert ctx.stats()["batch_blocks"] == 6 and all(np.array_equal(b, v) for b, v in zip(bs, xs))
        T = np.append(x[::-1], np.uint8(0x41))
        U = T.copy()
        LF = np.full(8, 0xDEAD, np.uint32)
        _expect_everify(lambda: ctx.divbwtf(U, U, LF, fr), "raw")
        assert np.array_equal(U, T) and (LF == 0xDEAD).all() and (fr == 3).all()
        # pipeline: 8 starting points fail, j do not
        items = []
        for k, starts in enumerate((j, 8, j)):
            xk = bw.generate("dna", n, seed=750 + k)
            b = xk.copy()
            items.append((starts, xk, b, p.submit(b, starts)))
        for starts, xk, b, h in items:
            if starts == 8:
                with pytest.raises(bw.BwtcCudaError) as ei:
                    p.wait(h)
                assert ei.value.code == bw.EVERIFY
                assert np.array_equal(b, xk)
            else:
                lf, _ = p.wait(h)
                want = oracle.block(xk, starts)
                assert np.array_equal(b, want[0]) and np.array_equal(lf, want[1])
    finally:
        ctx.close()
        p.close()


def test_wrong_starting_point_is_found_with_lazy_ranks(oracle, monkeypatch):
    """BWTC_LAZY=2: LFpowers come from the rank look-up in the sorted keys (not from the emission of the bytes); with them
    verification passes, a changed LFpowers[3] fails, for a block and a raw call."""
    monkeypatch.setenv("BWTC_LAZY", "2")
    n = 1 << 20
    good = bw.CudaContext(n + 1)
    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_LF", "3")
    bad = bw.CudaContext(n + 1)
    try:
        good.set_verify(True)
        bad.set_verify(True)
        x = bw.generate("dna", n, seed=760)
        T = raw_text(x)
        want_b = oracle.block(x, 8)
        got = good.bwt_block(x.copy(), np.zeros(8, np.uint32), None)
        assert got == want_b[1][0] and good.stats()["flags"] & F_LAZY and _verified(good)
        assert_raw(run_raw(good, T, 8), oracle.raw(T, 8), "lazy raw")
        assert good.stats()["flags"] & F_LAZY and _verified(good)
        blk = x.copy()
        _expect_everify(lambda: bad.bwt_block(blk, np.zeros(8, np.uint32), None), "lazy block")
        assert bad.stats()["flags"] & F_LAZY and np.array_equal(blk, x)
        U = T.copy()
        _expect_everify(lambda: bad.divbwtf(U, U, np.zeros(8, np.uint32), None), "lazy raw")
        assert np.array_equal(U, T)
    finally:
        good.close()
        bad.close()


# ---- verification off, the environment switch, the watchdog ----------------------------------------------------------
def test_verify_off_raw_runs_the_same_kernels(oracle):
    T = np.append(bw.generate("markov", (1 << 20) - 1, seed=770), np.uint8(0x61))
    a, b = bw.CudaContext(1 << 20), bw.CudaContext(1 << 20)
    try:
        b.set_verify(True)
        b.set_verify(False)
        ra, rb = run_raw(a, T, 8), run_raw(b, T, 8)
        sa, sb = a.stats(), b.stats()
        assert sa["kernel_launches"] == sb["kernel_launches"] and sa["algorithmic_bytes"] == sb["algorithmic_bytes"]
        assert not sb["flags"] & bw.FLAG_VERIFIED
        for u, v in zip(ra[1:], rb[1:]):
            assert np.array_equal(u, v)
        b.set_verify(True)
        rc = run_raw(b, T, 8)
        assert all(np.array_equal(u, v) for u, v in zip(ra[1:], rc[1:])) and rc[0] == ra[0]
        assert b.stats()["kernel_launches"] > sa["kernel_launches"] and _verified(b)
    finally:
        a.close()
        b.close()


def test_environment_switch(oracle, monkeypatch):
    """BWTC_VERIFY=1 before contexts and pipelines are created: block, batch, raw, pipeline and CudaBWTransform calls are
    verified without any set_verify call; set_verify(False) switches it off per context and per pipeline."""
    monkeypatch.setenv("BWTC_VERIFY", "1")
    n = 50000
    ctx = bw.CudaContext(8 * (n + 1))
    p = bw.Pipeline(n, depth=2)
    tr = bw.CudaBWTransform(n + 1)
    monkeypatch.delenv("BWTC_VERIFY")
    try:
        x = bw.generate("markov", n, seed=780)
        want = oracle.block(x, 8)
        blk = x.copy()
        LF = np.zeros(8, np.uint32)
        ctx.bwt_block(blk, LF, None)
        assert _verified(ctx) and np.array_equal(blk, want[0]) and np.array_equal(LF, want[1])
        xs = [bw.generate("dna", n, seed=781 + k) for k in range(4)]
        bs = [v.copy() for v in xs]
        ctx.bwt_blocks(bs, 8)
        assert _verified(ctx) and ctx.stats()["batch_blocks"] == 4
        assert all(np.array_equal(b, oracle.block(v, 8)[0]) for b, v in zip(bs, xs))
        T = np.append(x, np.uint8(0x30))
        assert_raw(run_raw(ctx, T, 8), oracle.raw(T, 8), "raw")
        assert _verified(ctx)
        U = T.copy()
        LF = np.zeros(8, np.uint32)
        assert tr.doTransformRaw(U, LF) == oracle.raw(T, 8)[0]
        assert tr.context.stats()["flags"] & bw.FLAG_VERIFIED
        blocks = [v.copy() for v in xs]
        _, _, _, stats = p.run(blocks, 8)
        assert all(s["flags"] & bw.FLAG_VERIFIED for s in stats)
        assert all(np.array_equal(b, oracle.block(v, 8)[0]) for b, v in zip(blocks, xs))
        ctx.set_verify(False)
        run_raw(ctx, T, 8)
        assert not _verified(ctx)
        ctx.bwt_block(x.copy(), np.zeros(8, np.uint32), None)
        assert not _verified(ctx)
        p.set_verify(False)
        _, _, _, stats = p.run([v.copy() for v in xs], 8)
        assert not any(s["flags"] & bw.FLAG_VERIFIED for s in stats)
    finally:
        ctx.close()
        p.close()
        tr.context.close()


def test_fake_watchdog_raw_verified(oracle, monkeypatch):
    """BWTC_DEBUG_FAKE_WATCHDOG=1 (the simulated look-back watchdog): a verified raw call repeats its sort with tile
    tickets and is exact."""
    monkeypatch.setenv("BWTC_DEBUG_FAKE_WATCHDOG", "1")
    ctx = bw.CudaContext(1 << 20)
    try:
        ctx.set_verify(True)
        T = np.append(bw.generate("dna", (1 << 20) - 1, seed=790), np.uint8(ord("G")))
        assert_raw(run_raw(ctx, T, 8), oracle.raw(T, 8), "fake watchdog")
        st = ctx.stats()
        assert st["flags"] & F_TICKETS and st["flags"] & bw.FLAG_VERIFIED
    finally:
        ctx.close()
