"""GPU tests of bwtc_cuda_divsufsort / _device and bwtc_cuda_sufcheck (DESIGN.md §3.11): the suffix array the forward
engine emits beside the BWT bytes, and the device-side check.  Every SA is compared with oracle_suffix_array
(oracle/oracle_bwt.c, the prefix-doubling oracle the forward tests are pinned on); sufcheck verdicts are compared with the
numpy restatement of tests/test_sufcheck_keys.py."""
import itertools

import numpy as np
import pytest

import bwtc_b200 as bw
from test_gpu_parity import ENGINE_KNOBS
from test_gpu_raw_contract import F_LAZY, F_TICKETS, KINDS
from test_sufcheck_keys import DUP, ORDER, RANGE, brute_sa, sufcheck


def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")]

MiB = 1 << 20
EARG, EALLOC, ETOOBIG = -1, -2, -5
SA_ENTRIES_PER_CHUNK = (4 << 20) // 4  # the pinned staging ring's 4 MiB chunk, in SA entries
REASONS = {RANGE: "out of range", DUP: "duplicate", ORDER: "out of order"}


def oracle_sa(oracle, T):
    if T.size == 0:
        return np.zeros(0, np.int32)
    SA, _ = oracle.suffix_array(np.ascontiguousarray(T))
    return SA.view(np.int32)


def inverse(SA):
    isa = np.empty(SA.size, np.int64)
    isa[SA] = np.arange(SA.size)
    return isa


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(8 * MiB)
    yield c
    c.close()


def check(ctx, T, want, what):
    SA = ctx.divsufsort(T)
    assert np.array_equal(SA, want), (what, int(np.count_nonzero(SA != want)))
    if T.size >= 2:
        assert ctx.stats()["flags"] & bw.FLAG_SA, what
    return SA


def check_against_bwt(ctx, T, SA, what):
    """divbwtf of the same text agrees with the SA: U[r] = T[SA[r]-1] (r != pidx), pidx = ISA[0], LFpowers[j] =
    ISA[n - j (n / 256)]."""
    n = T.size
    U = np.zeros(n, np.uint8)
    LF = np.zeros(256, np.uint32)
    pidx = ctx.divbwtf(T, U, LF, None)
    isa = inverse(SA)
    assert pidx == isa[0] == LF[0], what
    rows = np.flatnonzero(np.arange(n) != pidx)
    assert np.array_equal(U[rows], T[SA[rows] - 1]), what
    x = n // 256
    assert np.array_equal(LF[1:], isa[n - np.arange(1, 256) * x]), what


# ---- short texts ----------------------------------------------------------------------------------------------------
def test_every_short_text(ctx):
    """Every text of length 2-7 over {0, 1, 2} and over {0x00, 0xFF}; sufcheck accepts each SA."""
    for alphabet in ((0, 1, 2), (0x00, 0xFF)):
        for n in range(2, 8):
            for t in itertools.product(alphabet, repeat=n):
                T = np.array(t, np.uint8)
                SA = check(ctx, T, brute_sa(T), t)
                assert ctx.sufcheck(T, SA), t


def test_trivial_lengths(ctx):
    """n = 0: nothing is written; n = 1: SA[0] = 0; n = 2 in both orders and with equal bytes (libdivsufsort's own
    n <= 2 cases)."""
    SA = np.full(1, 77, np.int32)
    assert ctx._lib.bwtc_cuda_divsufsort(ctx._h, np.zeros(1, np.uint8).ctypes.data, SA.ctypes.data, 0) == 0
    assert SA[0] == 77
    assert ctx.divsufsort(np.array([9], np.uint8)).tolist() == [0]
    for t, want in (((1, 2), [0, 1]), ((2, 1), [1, 0]), ((5, 5), [1, 0]), ((0, 0), [1, 0])):
        check(ctx, np.array(t, np.uint8), np.array(want, np.int32), t)
    assert ctx.sufcheck(np.array([3], np.uint8), np.array([0], np.int32))
    assert not ctx.sufcheck(np.array([3], np.uint8), np.array([1], np.int32))
    assert ctx.sufcheck(np.zeros(0, np.uint8), np.zeros(0, np.int32))


# ---- the input families ---------------------------------------------------------------------------------------------
def _special(name, n, rng):
    if name == "one_byte":
        return np.full(n, 0x61, np.uint8)
    if name == "all_256":
        T = rng.integers(0, 256, n).astype(np.uint8)
        T[:256] = np.arange(256)
        return T
    if name == "zeros":
        T = np.zeros(n, np.uint8)
        T[rng.integers(0, n, n // 64)] = rng.integers(1, 4, n // 64)
        return T
    raise ValueError(name)


@pytest.mark.parametrize("size", [1 << 10, (64 << 10) + 3, MiB, 8 * MiB])
@pytest.mark.parametrize("kind", list(KINDS) + ["one_byte", "all_256", "zeros"])
def test_families(ctx, oracle, kind, size):
    """Every generator of bwtc_b200.generate, a single repeated byte (the most rounds), all 256 byte values, and text that
    is mostly 0x00, from 1 KiB to 8 MiB: SA = the oracle's, sufcheck accepts it, divbwtf of the same text agrees."""
    rng = np.random.default_rng(size)
    T = bw.generate(kind, size, seed=61) if kind in KINDS else _special(kind, size, rng)
    want = oracle_sa(oracle, T)
    SA = check(ctx, T, want, (kind, size))
    assert ctx.sufcheck(T, SA)
    check_against_bwt(ctx, T, SA, (kind, size))


@pytest.mark.parametrize("kind,mib", [("markov", 32), ("dna", 64)])
def test_large_texts(oracle, kind, mib):
    T = bw.generate(kind, mib * MiB, seed=62)
    c = bw.CudaContext(mib * MiB)
    try:
        SA = check(c, T, oracle_sa(oracle, T), kind)
        assert c.sufcheck(T, SA)
        check_against_bwt(c, T, SA, kind)
    finally:
        c.close()


# ---- every engine path ----------------------------------------------------------------------------------------------
_ENGINE_SA = {}


def _engine_cases(oracle):
    """About 2 MiB per family: with BWTC_RERANK_WINDOW_MB=1 the rank array spans 8 windows (bucketed scatter), with 4 or
    6 two windows (windowed relaunches)."""
    if not _ENGINE_SA:
        for i, kind in enumerate(KINDS):
            T = bw.generate(kind, 2 * MiB + 5 + i, seed=63)
            _ENGINE_SA[kind] = (T, oracle_sa(oracle, T))
    return _ENGINE_SA.items()


@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()) or "default")
def test_every_engine_path(oracle, monkeypatch, knobs):
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    tickets = knobs.get("BWTC_STATIC_TILES") == "0" or knobs.get("BWTC_DEBUG_FAKE_WATCHDOG") == "1"
    c = bw.CudaContext(4 * MiB)
    try:
        for kind, (T, want) in _engine_cases(oracle):
            check(c, T, want, (kind, knobs))
            st = c.stats()
            assert bool(st["flags"] & F_TICKETS) == tickets, (kind, st["flags"])
            if knobs.get("BWTC_LAZY") == "2":
                assert st["flags"] & F_LAZY, kind
            if knobs.get("BWTC_LAZY") == "0":
                assert not st["flags"] & F_LAZY, kind
    finally:
        c.close()


# ---- buffer kinds and limits ----------------------------------------------------------------------------------------
def _pinned(a):
    import torch

    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t, t.numpy()


def test_buffer_kinds(ctx, oracle):
    """Pageable, pinned and device T / SA; pageable T and SA at unaligned starts."""
    import torch

    T = bw.generate("markov", 3 * MiB + 7, seed=64)
    want = oracle_sa(oracle, T)
    n = T.size
    # pinned T and SA, in every combination with pageable ones
    tT, pT = _pinned(T)
    tS, pS = _pinned(np.zeros(n, np.int32))
    for TT in (T, pT):
        for SS in (np.zeros(n, np.int32), pS):
            SS[:] = -5
            ctx.divsufsort(TT, SS)
            assert np.array_equal(SS, want)
    # unaligned pageable starts
    for off in (1, 2, 3):
        bT = np.zeros(n + 8, np.uint8)
        TT = bT[off:off + n]
        TT[:] = T
        bS = np.zeros(4 * n + 8, np.uint8)
        SS = np.frombuffer(bS.data, dtype=np.int32, count=n, offset=off)
        ctx._check(ctx._lib.bwtc_cuda_divsufsort(ctx._h, TT.ctypes.data, SS.ctypes.data, n))
        assert np.array_equal(SS, want), off
        assert ctx.sufcheck(np.ascontiguousarray(TT), np.ascontiguousarray(SS))
    # device T and SA (torch), and a device SA at a 4-byte (not 16-byte) aligned offset
    dT = torch.from_numpy(T).cuda()
    dS = torch.full((n + 4,), -1, dtype=torch.int32, device="cuda")
    for off in (0, 1, 3):
        dS.fill_(-1)
        ctx.divsufsort_device(dT.data_ptr(), dS.data_ptr() + 4 * off, n)
        torch.cuda.synchronize()
        got = dS.cpu().numpy()
        assert np.array_equal(got[off:off + n], want), off
        assert (got[:off] == -1).all() and (got[off + n:] == -1).all(), off
        assert ctx.stats()["flags"] & bw.FLAG_SA
    # device n == 1
    dS.fill_(-1)
    ctx.divsufsort_device(dT.data_ptr(), dS.data_ptr(), 1)
    assert int(dS[0]) == 0


@pytest.mark.parametrize("n", [SA_ENTRIES_PER_CHUNK - 1, SA_ENTRIES_PER_CHUNK, SA_ENTRIES_PER_CHUNK + 1, 2 * SA_ENTRIES_PER_CHUNK])
def test_staging_ring_chunk_edges(ctx, oracle, n):
    """The SA is 4 bytes per suffix: pageable copies cross a staging-ring chunk every 1 Mi entries."""
    T = bw.generate("dna", n, seed=65)
    SA = np.full(n + 1, -3, np.int32)
    ctx.divsufsort(T, SA[:n])
    assert np.array_equal(SA[:n], oracle_sa(oracle, T)) and SA[n] == -3


def test_limits_and_argument_errors(oracle):
    """n = max_block_bytes + 1 succeeds, + 2 is ETOOBIG; null pointers and a misaligned d_SA are EARG; the context stays
    usable after each error."""
    import torch

    cap = 4096
    c = bw.CudaContext(cap)
    lib, h = c._lib, c._h
    try:
        T = bw.generate("markov", cap + 2, seed=66)
        ok = T[: cap + 1].copy()
        good = oracle_sa(oracle, ok)

        def still_usable():
            assert np.array_equal(c.divsufsort(ok), good)

        still_usable()
        SA = np.zeros(cap + 2, np.int32)
        assert lib.bwtc_cuda_divsufsort(h, T.ctypes.data, SA.ctypes.data, cap + 2) == ETOOBIG
        still_usable()
        assert lib.bwtc_cuda_sufcheck(h, T.ctypes.data, SA.ctypes.data, cap + 2) == ETOOBIG
        still_usable()
        assert lib.bwtc_cuda_divsufsort(h, None, SA.ctypes.data, 10) == EARG
        assert lib.bwtc_cuda_divsufsort(h, T.ctypes.data, None, 10) == EARG
        assert lib.bwtc_cuda_sufcheck(h, None, SA.ctypes.data, 10) == EARG
        assert lib.bwtc_cuda_sufcheck(h, T.ctypes.data, None, 10) == EARG
        assert lib.bwtc_cuda_divsufsort(None, T.ctypes.data, SA.ctypes.data, 10) == EARG
        still_usable()
        dT = torch.from_numpy(ok).cuda()
        dS = torch.zeros(cap + 4, dtype=torch.int32, device="cuda")
        assert lib.bwtc_cuda_divsufsort_device(h, None, dS.data_ptr(), 10) == EARG
        assert lib.bwtc_cuda_divsufsort_device(h, dT.data_ptr(), None, 10) == EARG
        assert lib.bwtc_cuda_divsufsort_device(h, dT.data_ptr(), dS.data_ptr() + 2, 10) == EARG
        assert lib.bwtc_cuda_divsufsort_device(h, dT.data_ptr(), dS.data_ptr(), cap + 2) == ETOOBIG
        still_usable()
        c.divsufsort_device(dT.data_ptr(), dS.data_ptr(), cap + 1)
        torch.cuda.synchronize()
        assert np.array_equal(dS[: cap + 1].cpu().numpy(), good)
    finally:
        c.close()


# ---- nothing leaks into the other entry points ----------------------------------------------------------------------
def _other_calls(c, T, x, blocks):
    U = np.zeros(T.size, np.uint8)
    LF = np.zeros(256, np.uint32)
    fr = np.zeros(256, np.uint32)
    out = [("divbwtf", c.divbwtf(T, U, LF, fr), U.copy(), LF.copy(), fr.copy())]
    st = c.stats()
    out.append(("divbwtf stats", st["kernel_launches"], st["flags"]))
    b = x.copy()
    LF2 = np.zeros(8, np.uint32)
    out.append(("bwt_block", c.bwt_block(b, LF2, None), b, LF2.copy()))
    st = c.stats()
    out.append(("bwt_block stats", st["kernel_launches"], st["flags"]))
    bl = [y.copy() for y in blocks]
    LF3, nLF3, fr3 = c.bwt_blocks(bl, 8)
    out.append(("bwt_blocks", [y.tobytes() for y in bl], LF3.copy(), nLF3.copy(), fr3.copy()))
    st = c.stats()
    out.append(("bwt_blocks stats", st["kernel_launches"], st["flags"]))
    return out


def _same(a, b):
    assert len(a) == len(b)
    for p, q in zip(a, b):
        assert p[0] == q[0]
        for u, v in zip(p[1:], q[1:]):
            if isinstance(u, np.ndarray):
                assert np.array_equal(u, v), p[0]
            else:
                assert u == v, (p[0], u, v)


def test_no_leakage_into_other_calls(oracle):
    """After divsufsort (host and device) on a context, divbwtf, bwt_block and bwt_blocks give the same bytes, launch
    counts and flags (bit 8 clear) as on a fresh context, and a device SA buffer they could reach stays untouched."""
    import torch

    T = bw.generate("markov", MiB + 3, seed=67)
    x = bw.generate("dna", 300000, seed=68)
    blocks = [bw.generate("random", 5000, seed=69 + k) for k in range(5)]
    fresh = bw.CudaContext(2 * MiB)
    try:
        want = _other_calls(fresh, T, x, blocks)
    finally:
        fresh.close()
    c = bw.CudaContext(2 * MiB)
    try:
        c.divsufsort(T)
        dT = torch.from_numpy(T).cuda()
        dS = torch.zeros(T.size, dtype=torch.int32, device="cuda")
        c.divsufsort_device(dT.data_ptr(), dS.data_ptr(), T.size)
        torch.cuda.synchronize()
        assert np.array_equal(dS.cpu().numpy(), oracle_sa(oracle, T))
        dS.fill_(0x5A5A5A5A)
        got = _other_calls(c, T, x, blocks)
        torch.cuda.synchronize()
        _same(got, want)
        for g in got:
            if g[0].endswith("stats"):
                assert not g[2] & bw.FLAG_SA, g
        assert (dS.cpu().numpy() == 0x5A5A5A5A).all()
    finally:
        c.close()


# ---- sufcheck --------------------------------------------------------------------------------------------------------
def _corruptions(T, SA, rng):
    n = SA.size
    out = []
    for r in (0, n // 2, n - 2):
        m = SA.copy()
        m[r], m[r + 1] = m[r + 1], m[r]
        out.append((f"swap {r}", m))
    for v in (n, -1):
        m = SA.copy()
        m[int(rng.integers(n))] = v
        out.append((f"value {v}", m))
    m = SA.copy()
    m[n // 3] = SA[n // 5]
    out.append(("duplicate", m))
    out.append(("rotation", np.roll(SA, 1)))
    return out


@pytest.mark.parametrize("kind", KINDS)
def test_sufcheck_rejects_corruptions(ctx, oracle, kind):
    """Adjacent swaps at r = 0, in the middle and at n - 2, the values n and -1, a duplicate, a rotation of the whole array
    (and, on repetitive text, swaps inside long repeats): rejected, with the row and reason the CPU restatement gives named
    in the message."""
    rng = np.random.default_rng(70)
    T = bw.generate(kind, 200003, seed=71)
    SA = oracle_sa(oracle, T)
    assert ctx.sufcheck(T, SA)
    cases = _corruptions(T, SA, rng)
    if kind == "repetitive":  # rows whose suffixes share a long prefix (the repeats): only the successor ranks differ
        lcp_like = [r for r in range(1, SA.size - 1)
                    if SA[r] + 64 < T.size and SA[r + 1] + 64 < T.size and
                    np.array_equal(T[SA[r]:SA[r] + 64], T[SA[r + 1]:SA[r + 1] + 64])]
        assert len(lcp_like) > 10
        for r in lcp_like[:: max(1, len(lcp_like) // 5)]:
            m = SA.copy()
            m[r], m[r + 1] = m[r + 1], m[r]
            cases.append((f"repeat swap {r}", m))
    for what, m in cases:
        want = sufcheck(T, m)
        assert want is not None, what
        assert not ctx.sufcheck(T, m), what
        msg = ctx.last_error()
        assert f"row {want[0]} " in msg and REASONS[want[1]] in msg, (what, want, msg)


def test_sufcheck_verdicts_equal_the_restatement(ctx):
    """Random short texts and random mutants: the device's verdict and row equal the numpy restatement's."""
    rng = np.random.default_rng(72)
    for trial in range(200):
        n = int(rng.integers(2, 3000))
        T = rng.integers(0, int(rng.choice([1, 2, 4, 256])), n).astype(np.uint8)
        SA = brute_sa(T) if n < 400 else ctx.divsufsort(T)
        m = SA.copy()
        k = int(rng.integers(4))
        if k == 0:
            i, j = rng.integers(n, size=2)
            m[i], m[j] = m[j], m[i]
        elif k == 1:
            m[int(rng.integers(n))] = int(rng.integers(-2, n + 2))
        elif k == 2:
            m = np.roll(m, int(rng.integers(n)))
        want = sufcheck(T, m)
        assert ctx.sufcheck(T, m) == (want is None), (trial, want)
        if want is not None:
            assert f"row {want[0]} " in ctx.last_error(), (trial, want, ctx.last_error())


# ---- verification ----------------------------------------------------------------------------------------------------
def test_verified_results_are_unchanged(ctx, oracle, monkeypatch):
    """set_verify(1) and BWTC_VERIFY=1: the same SA, flags bits 6 and 8 set."""
    import torch

    T = bw.generate("markov", 2 * MiB + 1, seed=73)
    want = oracle_sa(oracle, T)
    ctx.set_verify(True)
    try:
        assert np.array_equal(ctx.divsufsort(T), want)
        assert ctx.stats()["flags"] & bw.FLAG_VERIFIED and ctx.stats()["flags"] & bw.FLAG_SA
    finally:
        ctx.set_verify(False)
    assert np.array_equal(ctx.divsufsort(T), want)
    assert not ctx.stats()["flags"] & bw.FLAG_VERIFIED
    monkeypatch.setenv("BWTC_VERIFY", "1")
    c = bw.CudaContext(4 * MiB)
    try:
        assert np.array_equal(c.divsufsort(T), want)
        assert c.stats()["flags"] & bw.FLAG_VERIFIED
        dT = torch.from_numpy(T).cuda()
        dS = torch.zeros(T.size, dtype=torch.int32, device="cuda")
        c.divsufsort_device(dT.data_ptr(), dS.data_ptr(), T.size)
        torch.cuda.synchronize()
        assert np.array_equal(dS.cpu().numpy(), want) and c.stats()["flags"] & bw.FLAG_VERIFIED
    finally:
        c.close()


@pytest.mark.parametrize("row", ["0", "1000", "last"])
def test_corrupt_sa_hook_gives_everify(oracle, monkeypatch, row):
    """BWTC_DEBUG_CORRUPT_SA=r swaps SA[r] and SA[r+1] on the device before the check: EVERIFY, pageable and pinned SA keep
    their previous contents, and the next call (verification off) succeeds."""
    T = bw.generate("dna", MiB + 11, seed=74)
    n = T.size
    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_SA", str(n - 2) if row == "last" else row)
    c = bw.CudaContext(2 * MiB)
    try:
        c.set_verify(True)
        _, pinned = _pinned(np.full(n, 123, np.int32))
        for SA in (np.full(n, 123, np.int32), pinned):
            with pytest.raises(bw.BwtcCudaError) as ei:
                c.divsufsort(T, SA)
            assert ei.value.code == bw.EVERIFY
            assert (SA == 123).all()
            assert c.stats()["flags"] & bw.FLAG_VERIFIED
        c.set_verify(False)
        assert np.array_equal(c.divsufsort(T), oracle_sa(oracle, T))
    finally:
        c.close()


def test_watchdog_retry_gives_the_same_sa(oracle, monkeypatch):
    """BWTC_DEBUG_FAKE_WATCHDOG=1: phase B is repeated with tile tickets and the SA is simply written again."""
    monkeypatch.setenv("BWTC_DEBUG_FAKE_WATCHDOG", "1")
    T = bw.generate("repetitive", 3 * MiB, seed=75)
    c = bw.CudaContext(4 * MiB)
    try:
        c.set_verify(True)
        assert np.array_equal(c.divsufsort(T), oracle_sa(oracle, T))
        assert c.stats()["flags"] & F_TICKETS and c.stats()["flags"] & bw.FLAG_VERIFIED
    finally:
        c.close()
