"""GPU tests of bwtc_cuda_divsufsort_lcp / _lcp_device (DESIGN.md §3.12): the suffix array and its LCP array, built on
the device behind the sort.  SAs are compared with divsufsort's (itself pinned on the prefix-doubling oracle by
tests/test_gpu_divsufsort.py) or brute force; LCPs with oracle_lcp (a sequential Kasai, tests/lcp_oracle.c), brute force,
or a closed form."""
import itertools

import numpy as np
import pytest

import bwtc_b200 as bw
from test_gpu_divsufsort import _pinned, _special, oracle_sa
from test_gpu_parity import ENGINE_KNOBS
from test_gpu_raw_contract import F_TICKETS, KINDS
from test_lcp_keys import LCP_SEG_BYTES, LCP_SHORT_BYTES, brute_lcp, oracle_lcp
from test_sufcheck_keys import brute_sa


def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")]

MiB = 1 << 20
EARG, ETOOBIG = -1, -5
ENTRIES_PER_CHUNK = (4 << 20) // 4  # the pinned staging ring's 4 MiB chunk, in int32 entries


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(8 * MiB)
    yield c
    c.close()


def check(ctx, T, want_sa, want_lcp, what):
    SA, LCP = ctx.divsufsort_lcp(T)
    assert np.array_equal(SA, want_sa), (what, int(np.count_nonzero(SA != want_sa)))
    assert np.array_equal(LCP, want_lcp), (what, np.flatnonzero(LCP != want_lcp)[:8].tolist())
    if T.size >= 2:
        fl = ctx.stats()["flags"]
        assert fl & bw.FLAG_SA and fl & bw.FLAG_LCP, (what, fl)
    return SA, LCP


# ---- short texts and trivial lengths --------------------------------------------------------------------------------
def test_every_short_text(ctx):
    for alphabet in ((0, 1, 2), (0x00, 0xFF)):
        for n in range(2, 8):
            for t in itertools.product(alphabet, repeat=n):
                T = np.array(t, np.uint8)
                SA = brute_sa(T)
                check(ctx, T, SA, brute_lcp(T, SA), t)


def test_trivial_lengths(ctx):
    """n = 0 writes nothing; n = 1 gives SA = LCP = [0] without the device (the stats of the previous call stay); n = 2 in
    both byte orders and with equal bytes."""
    lib, h = ctx._lib, ctx._h
    SA, LCP = np.full(1, 77, np.int32), np.full(1, 78, np.int32)
    assert lib.bwtc_cuda_divsufsort_lcp(h, np.zeros(1, np.uint8).ctypes.data, SA.ctypes.data, LCP.ctypes.data, 0) == 0
    assert SA[0] == 77 and LCP[0] == 78
    ctx.divsufsort_lcp(np.array([4, 3, 4], np.uint8))
    before = ctx.stats()
    SA, LCP = ctx.divsufsort_lcp(np.array([9], np.uint8))
    assert SA.tolist() == [0] and LCP.tolist() == [0]
    after = ctx.stats()
    assert all(after[k] == before[k] for k in ("kernel_launches", "flags", "gpu_ms", "n_suffixes"))
    for t, sa, lcp in (((1, 2), [0, 1], [0, 0]), ((2, 1), [1, 0], [0, 0]), ((5, 5), [1, 0], [0, 1]),
                       ((0, 0), [1, 0], [0, 1])):
        check(ctx, np.array(t, np.uint8), np.array(sa, np.int32), np.array(lcp, np.int32), t)


# ---- families and large texts ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", [1 << 10, (64 << 10) + 3, MiB, 8 * MiB])
@pytest.mark.parametrize("kind", list(KINDS) + ["one_byte", "all_256", "zeros"])
def test_families(ctx, oracle, kind, size):
    rng = np.random.default_rng(size)
    T = bw.generate(kind, size, seed=81) if kind in KINDS else _special(kind, size, rng)
    want_sa = ctx.divsufsort(T)
    check(ctx, T, want_sa, oracle_lcp(T, want_sa), (kind, size))


@pytest.mark.parametrize("kind,mib", [("markov", 32), ("dna", 64)])
def test_large_texts(oracle, kind, mib):
    T = bw.generate(kind, mib * MiB, seed=82)
    c = bw.CudaContext(mib * MiB)
    try:
        want_sa = oracle_sa(oracle, T)
        check(c, T, want_sa, oracle_lcp(T, want_sa), kind)
    finally:
        c.close()


def test_one_byte_256_mib():
    """A single repeated byte: one irreducible comparison of n - 1 bytes, spread over the windows.  SA[r] = n-1-r,
    LCP[r] = r."""
    n = 256 * MiB
    T = np.full(n, 0x61, np.uint8)
    c = bw.CudaContext(n)
    try:
        SA, LCP = c.divsufsort_lcp(T)
        r = np.arange(n, dtype=np.int64)
        assert np.array_equal(SA, (n - 1 - r).astype(np.int32))
        assert np.array_equal(LCP, r.astype(np.int32))
        assert c.stats()["flags"] & bw.FLAG_LCP
    finally:
        c.close()


# ---- tier edges -----------------------------------------------------------------------------------------------------
def _edge_lengths():
    K, out = LCP_SHORT_BYTES, set()
    for edge in (K, 2 * K, 4 * K, LCP_SEG_BYTES, 2 * LCP_SEG_BYTES, 4 * LCP_SEG_BYTES):
        out |= {edge - 1, edge, edge + 1}
    return sorted(out)


@pytest.mark.parametrize("ell", _edge_lengths())
def test_tier_edges(ctx, oracle, ell):
    """Two copies of a random string of length ell in random text: their suffixes share exactly ell bytes (the bytes
    before and after the copies differ), and that irreducible pair resolves at ell: at the short tier's end, at each window
    edge, and at the segment edges of the windows."""
    rng = np.random.default_rng(ell)
    n = 64 * 1024 + 3 * ell
    T = rng.integers(0, 256, n).astype(np.uint8)
    s = rng.integers(0, 256, ell).astype(np.uint8)
    p, q = 1000, n // 2 + 17
    T[p:p + ell] = s
    T[q:q + ell] = s
    T[q - 1] = T[p - 1] ^ 1
    T[q + ell] = T[p + ell] ^ 1
    want_sa = ctx.divsufsort(T)
    want = oracle_lcp(T, want_sa)
    _, LCP = check(ctx, T, want_sa, want, ell)
    isa = np.empty(n, np.int64)
    isa[want_sa] = np.arange(n)
    r = max(isa[p], isa[q])
    assert abs(isa[p] - isa[q]) == 1 and LCP[r] == ell


# ---- every engine path ----------------------------------------------------------------------------------------------
_ENGINE = {}


def _engine_cases(oracle):
    if not _ENGINE:
        for i, kind in enumerate(KINDS):
            T = bw.generate(kind, 2 * MiB + 5 + i, seed=83)
            sa = oracle_sa(oracle, T)
            _ENGINE[kind] = (T, sa, oracle_lcp(T, sa))
    return _ENGINE.items()


@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()) or "default")
def test_every_engine_path(oracle, monkeypatch, knobs):
    """Whatever buffers the sort's path leaves behind, the LCP stage reads the SA and the text correctly."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    tickets = knobs.get("BWTC_STATIC_TILES") == "0" or knobs.get("BWTC_DEBUG_FAKE_WATCHDOG") == "1"
    c = bw.CudaContext(4 * MiB)
    try:
        for kind, (T, sa, lcp) in _engine_cases(oracle):
            check(c, T, sa, lcp, (kind, knobs))
            assert bool(c.stats()["flags"] & F_TICKETS) == tickets, kind
    finally:
        c.close()


# ---- buffer kinds ---------------------------------------------------------------------------------------------------
def test_host_buffer_kinds(ctx, oracle):
    """Pageable and pinned SA / LCP in all four combinations."""
    T = bw.generate("markov", 3 * MiB + 7, seed=84)
    want_sa = ctx.divsufsort(T)
    want = oracle_lcp(T, want_sa)
    n = T.size
    _, pS = _pinned(np.zeros(n, np.int32))
    _, pL = _pinned(np.zeros(n, np.int32))
    for SS in (np.zeros(n, np.int32), pS):
        for LL in (np.zeros(n, np.int32), pL):
            SS[:] = -5
            LL[:] = -6
            ctx.divsufsort_lcp(T, SS, LL)
            assert np.array_equal(SS, want_sa) and np.array_equal(LL, want)


@pytest.mark.parametrize("n", [ENTRIES_PER_CHUNK - 1, ENTRIES_PER_CHUNK, ENTRIES_PER_CHUNK + 1])
def test_staging_ring_chunk_edges(ctx, oracle, n):
    T = bw.generate("dna", n, seed=85)
    SA = np.full(n + 1, -3, np.int32)
    LCP = np.full(n + 1, -4, np.int32)
    ctx.divsufsort_lcp(T, SA[:n], LCP[:n])
    assert SA[n] == -3 and LCP[n] == -4
    assert np.array_equal(SA[:n], ctx.divsufsort(T))
    assert np.array_equal(LCP[:n], oracle_lcp(T, SA[:n]))


def test_device_buffers(ctx, oracle):
    """Torch tensors; d_T at byte offsets 1 and 3 and as the last n bytes of its tensor; misaligned or overlapping d_SA /
    d_LCP are EARG and leave both untouched."""
    import torch

    T = bw.generate("repetitive", MiB + 13, seed=86)
    n = T.size
    want_sa = ctx.divsufsort(T)
    want = oracle_lcp(T, want_sa)
    dS = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    dL = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    for off in (0, 1, 3):
        buf = torch.zeros(n + 8, dtype=torch.uint8, device="cuda")
        buf[off:off + n] = torch.from_numpy(T).cuda()
        dS.fill_(-1)
        dL.fill_(-1)
        ctx.divsufsort_lcp_device(buf.data_ptr() + off, dS.data_ptr(), dL.data_ptr(), n)
        torch.cuda.synchronize()
        assert np.array_equal(dS.cpu().numpy(), want_sa) and np.array_equal(dL.cpu().numpy(), want), off
        assert ctx.stats()["flags"] & bw.FLAG_LCP
    tail = torch.zeros(n + 5, dtype=torch.uint8, device="cuda")
    tail[5:] = torch.from_numpy(T).cuda()
    ctx.divsufsort_lcp_device(tail.data_ptr() + 5, dS.data_ptr(), dL.data_ptr(), n)
    torch.cuda.synchronize()
    assert np.array_equal(dL.cpu().numpy(), want)
    lib, h = ctx._lib, ctx._h
    big = torch.full((2 * n + 8,), -7, dtype=torch.int32, device="cuda")
    dT = torch.from_numpy(T).cuda()
    bad = [(big.data_ptr() + 2, big.data_ptr() + 4 * (n + 4)),          # misaligned d_SA
           (big.data_ptr(), big.data_ptr() + 4 * (n + 4) + 1),           # misaligned d_LCP
           (big.data_ptr(), big.data_ptr() + 4 * (n - 1)),               # d_LCP starts inside d_SA
           (big.data_ptr() + 4 * 8, big.data_ptr()),                     # d_SA starts inside d_LCP
           (big.data_ptr(), big.data_ptr())]
    for a, b in bad:
        assert lib.bwtc_cuda_divsufsort_lcp_device(h, dT.data_ptr(), a, b, n) == EARG, (a, b)
    torch.cuda.synchronize()
    assert (big.cpu().numpy() == -7).all()
    ctx.divsufsort_lcp_device(dT.data_ptr(), big.data_ptr(), big.data_ptr() + 4 * n, n)  # adjacent: fine
    torch.cuda.synchronize()
    assert np.array_equal(big[n:2 * n].cpu().numpy(), want)
    # n == 1 on the device
    dS.fill_(-1)
    dL.fill_(-1)
    ctx.divsufsort_lcp_device(dT.data_ptr(), dS.data_ptr(), dL.data_ptr(), 1)
    assert int(dS[0]) == 0 and int(dL[0]) == 0 and int(dS[1]) == -1


# ---- limits and flags -----------------------------------------------------------------------------------------------
def test_limits_and_argument_errors(oracle):
    import torch

    cap = 4096
    c = bw.CudaContext(cap)
    lib, h = c._lib, c._h
    try:
        T = bw.generate("markov", cap + 2, seed=87)
        ok = T[: cap + 1].copy()
        good_sa = oracle_sa(oracle, ok)
        good = oracle_lcp(ok, good_sa)

        def still_usable():
            SA, LCP = c.divsufsort_lcp(ok)
            assert np.array_equal(SA, good_sa) and np.array_equal(LCP, good)

        still_usable()
        SA = np.zeros(cap + 2, np.int32)
        LCP = np.zeros(cap + 2, np.int32)
        assert lib.bwtc_cuda_divsufsort_lcp(h, T.ctypes.data, SA.ctypes.data, LCP.ctypes.data, cap + 2) == ETOOBIG
        still_usable()
        assert lib.bwtc_cuda_divsufsort_lcp(h, None, SA.ctypes.data, LCP.ctypes.data, 10) == EARG
        assert lib.bwtc_cuda_divsufsort_lcp(h, T.ctypes.data, None, LCP.ctypes.data, 10) == EARG
        assert lib.bwtc_cuda_divsufsort_lcp(h, T.ctypes.data, SA.ctypes.data, None, 10) == EARG
        assert lib.bwtc_cuda_divsufsort_lcp(None, T.ctypes.data, SA.ctypes.data, LCP.ctypes.data, 10) == EARG
        assert (SA == 0).all() and (LCP == 0).all()
        dT = torch.from_numpy(ok).cuda()
        dS = torch.zeros(cap + 4, dtype=torch.int32, device="cuda")
        dL = torch.zeros(cap + 4, dtype=torch.int32, device="cuda")
        assert lib.bwtc_cuda_divsufsort_lcp_device(h, None, dS.data_ptr(), dL.data_ptr(), 10) == EARG
        assert lib.bwtc_cuda_divsufsort_lcp_device(h, dT.data_ptr(), None, dL.data_ptr(), 10) == EARG
        assert lib.bwtc_cuda_divsufsort_lcp_device(h, dT.data_ptr(), dS.data_ptr(), None, 10) == EARG
        assert lib.bwtc_cuda_divsufsort_lcp_device(h, dT.data_ptr(), dS.data_ptr(), dL.data_ptr(), cap + 2) == ETOOBIG
        still_usable()
        c.divsufsort_lcp_device(dT.data_ptr(), dS.data_ptr(), dL.data_ptr(), cap + 1)
        torch.cuda.synchronize()
        assert np.array_equal(dL[: cap + 1].cpu().numpy(), good)
    finally:
        c.close()


def _other_calls(c, T, x):
    """divsufsort, divbwtf, bwt_block and inverse_block: results, launch counts and flags."""
    out = [("divsufsort", c.divsufsort(T).copy())]
    st = c.stats()
    out.append(("divsufsort stats", st["kernel_launches"], st["flags"]))
    U = np.zeros(T.size, np.uint8)
    LF = np.zeros(256, np.uint32)
    fr = np.zeros(256, np.uint32)
    out.append(("divbwtf", c.divbwtf(T, U, LF, fr), U.copy(), LF.copy(), fr.copy()))
    st = c.stats()
    out.append(("divbwtf stats", st["kernel_launches"], st["flags"]))
    b = x.copy()
    LF2 = np.zeros(8, np.uint32)
    out.append(("bwt_block", c.bwt_block(b, LF2, None), b.copy(), LF2.copy()))
    st = c.stats()
    out.append(("bwt_block stats", st["kernel_launches"], st["flags"]))
    c.inverse_block(b, LF2)
    assert np.array_equal(b, x)
    out.append(("inverse_block", b.copy()))
    st = c.stats()
    out.append(("inverse_block stats", st["kernel_launches"], st["flags"]))
    return out


def test_flags_and_no_leakage(oracle):
    """Interleaved with divsufsort_lcp on one context, the other calls give a fresh context's results, launch counts and
    flags (bit 9 clear); divsufsort_lcp gives the same results between them; scratch_bytes is unchanged."""
    T = bw.generate("markov", MiB + 3, seed=88)
    x = bw.generate("dna", 300000, seed=89)
    cap = 2 * MiB
    scratch = bw.load_library().bwtc_cuda_scratch_bytes(cap)
    fresh = bw.CudaContext(cap)
    try:
        want = _other_calls(fresh, T, x)
        want_sa, want_lcp = fresh.divsufsort_lcp(T)
    finally:
        fresh.close()
    for g in want:
        if g[0].endswith("stats"):
            assert not g[2] & bw.FLAG_LCP, g
    c = bw.CudaContext(cap)
    try:
        for _ in range(2):
            SA, LCP = c.divsufsort_lcp(T)
            assert np.array_equal(SA, want_sa) and np.array_equal(LCP, want_lcp)
            assert c.stats()["flags"] & bw.FLAG_SA and c.stats()["flags"] & bw.FLAG_LCP
            got = _other_calls(c, T, x)
            assert len(got) == len(want)
            for p, q in zip(got, want):
                assert p[0] == q[0]
                for u, v in zip(p[1:], q[1:]):
                    assert np.array_equal(u, v) if isinstance(u, np.ndarray) else u == v, (p[0], u, v)
        assert bw.load_library().bwtc_cuda_scratch_bytes(cap) == scratch
        assert np.array_equal(oracle_lcp(T, want_sa), want_lcp)
    finally:
        c.close()


# ---- verification and the watchdog ----------------------------------------------------------------------------------
def test_verified_results_are_unchanged(ctx, oracle):
    T = bw.generate("dna", 2 * MiB + 1, seed=90)
    want_sa, want = ctx.divsufsort_lcp(T)
    assert np.array_equal(want, oracle_lcp(T, want_sa))
    ctx.set_verify(True)
    try:
        SA, LCP = ctx.divsufsort_lcp(T)
        fl = ctx.stats()["flags"]
        assert fl & bw.FLAG_VERIFIED and fl & bw.FLAG_SA and fl & bw.FLAG_LCP
        assert np.array_equal(SA, want_sa) and np.array_equal(LCP, want)
    finally:
        ctx.set_verify(False)


@pytest.mark.parametrize("row", ["0", "last"])
def test_corrupt_sa_hook_gives_everify(oracle, monkeypatch, row):
    """BWTC_DEBUG_CORRUPT_SA=r: EVERIFY, and pageable / pinned SA and LCP keep their previous contents."""
    T = bw.generate("markov", MiB + 11, seed=91)
    n = T.size
    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_SA", str(n - 2) if row == "last" else row)
    c = bw.CudaContext(2 * MiB)
    try:
        c.set_verify(True)
        _, pS = _pinned(np.full(n, 123, np.int32))
        _, pL = _pinned(np.full(n, 321, np.int32))
        for SA, LCP in ((np.full(n, 123, np.int32), np.full(n, 321, np.int32)), (pS, pL)):
            with pytest.raises(bw.BwtcCudaError) as ei:
                c.divsufsort_lcp(T, SA, LCP)
            assert ei.value.code == bw.EVERIFY
            assert (SA == 123).all() and (LCP == 321).all()
        c.set_verify(False)
        SA, LCP = c.divsufsort_lcp(T)
        assert np.array_equal(LCP, oracle_lcp(T, SA))
    finally:
        c.close()


def test_watchdog_retry_gives_the_same_arrays(oracle, monkeypatch):
    T = bw.generate("repetitive", 3 * MiB, seed=92)
    want_sa = oracle_sa(oracle, T)
    want = oracle_lcp(T, want_sa)
    monkeypatch.setenv("BWTC_DEBUG_FAKE_WATCHDOG", "1")
    c = bw.CudaContext(4 * MiB)
    try:
        SA, LCP = c.divsufsort_lcp(T)
        assert np.array_equal(SA, want_sa) and np.array_equal(LCP, want)
        assert c.stats()["flags"] & F_TICKETS and c.stats()["flags"] & bw.FLAG_LCP
    finally:
        c.close()
