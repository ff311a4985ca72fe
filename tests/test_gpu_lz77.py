"""GPU tests of bwtc_cuda_lz77 / _device (DESIGN.md §3.14): the greedy LZ77 factorisation, computed on the device from the
suffix and LCP arrays behind the sort.  Every result is compared bit for bit, src and len, with oracle_lz77 (the
sequential parse of tests/lz77_oracle.c, pinned to brute force by tests/test_lz77_keys.py) or a closed form, and decoded
back to the text."""
import itertools

import numpy as np
import pytest

import bwtc_b200 as bw
from test_gpu_divsufsort import _pinned, _special, oracle_sa
from test_gpu_parity import ENGINE_KNOBS
from test_gpu_raw_contract import F_TICKETS, KINDS
from test_lz77_keys import LZ_GROUP, LZ_ROW_TILE, LZ_TEXT_TILE, brute_lz77, decode, oracle_lz77
from test_sufcheck_keys import brute_sa


def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")]

MiB = 1 << 20
EARG, ETOOBIG = -1, -5


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(8 * MiB)
    yield c
    c.close()


def check(ctx, T, want_src, want_len, what):
    src, ln = ctx.lz77(T)
    assert np.array_equal(ln, want_len), (what, src.size, want_src.size, np.flatnonzero(ln[:want_len.size] != want_len[:ln.size])[:8].tolist())
    assert np.array_equal(src, want_src), (what, np.flatnonzero(src != want_src)[:8].tolist())
    assert np.array_equal(decode(src, ln, T.size), T), what
    if T.size >= 2:
        fl = ctx.stats()["flags"]
        assert fl & bw.FLAG_SA and fl & bw.FLAG_LCP and fl & bw.FLAG_LZ77, (what, fl)
    return src, ln


def with_oracle(ctx, T, what, SA=None):
    SA = ctx.divsufsort(T) if SA is None else SA
    return check(ctx, T, *oracle_lz77(T, SA), what)


def lz_counters(c):
    """debug_read(11): phrases, rows outside their tile, HBM rounds that found new starts."""
    u64 = c.debug_read(11, np.uint64, 2)
    return int(u64[0]), int(u64[1]), int(c.debug_read(11, np.uint32, 1, 16)[0])


# ---- short texts and trivial lengths --------------------------------------------------------------------------------
def test_every_short_text(ctx):
    for alphabet in ((0, 1, 2), (0x00, 0xFF)):
        for n in range(2, 8):
            for t in itertools.product(alphabet, repeat=n):
                T = np.array(t, np.uint8)
                check(ctx, T, *brute_lz77(T), t)


def test_trivial_lengths(ctx):
    """n = 0 returns 0 and writes nothing; n = 1 returns the literal without the device (the stats of the previous call
    stay); n = 2 in both byte orders and with equal bytes."""
    lib, h = ctx._lib, ctx._h
    src, ln = np.full(2, 77, np.int32), np.full(2, 78, np.int32)
    assert lib.bwtc_cuda_lz77(h, np.zeros(1, np.uint8).ctypes.data, 0, src.ctypes.data, ln.ctypes.data, 2) == 0
    assert (src == 77).all() and (ln == 78).all()
    ctx.lz77(np.array([4, 3, 4], np.uint8))
    before = ctx.stats()
    assert lib.bwtc_cuda_lz77(h, np.array([9], np.uint8).ctypes.data, 1, None, None, 0) == 1
    s, l = ctx.lz77(np.array([9], np.uint8))
    assert s.tolist() == [9] and l.tolist() == [0]
    after = ctx.stats()
    assert all(after[k] == before[k] for k in ("kernel_launches", "flags", "gpu_ms", "n_suffixes"))
    for t, want in (((1, 2), [(1, 0), (2, 0)]), ((2, 1), [(2, 0), (1, 0)]), ((5, 5), [(5, 0), (0, 1)]),
                    ((0, 0), [(0, 0), (0, 1)])):
        check(ctx, np.array(t, np.uint8), np.array([w[0] for w in want], np.int32), np.array([w[1] for w in want], np.int32), t)


# ---- families and large texts ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", [1 << 10, (64 << 10) + 3, MiB, 8 * MiB])
@pytest.mark.parametrize("kind", list(KINDS) + ["one_byte", "all_256", "zeros"])
def test_families(ctx, kind, size):
    rng = np.random.default_rng(size)
    T = bw.generate(kind, size, seed=101) if kind in KINDS else _special(kind, size, rng)
    with_oracle(ctx, T, (kind, size))


@pytest.mark.parametrize("kind,mib", [("markov", 32), ("dna", 64)])
def test_large_texts(oracle, kind, mib):
    T = bw.generate(kind, mib * MiB, seed=102)
    c = bw.CudaContext(mib * MiB)
    try:
        with_oracle(c, T, kind, oracle_sa(oracle, T))
    finally:
        c.close()


def test_one_byte_256_mib():
    """A single repeated byte: a literal, then one phrase of n - 1 bytes from position 0."""
    n = 256 * MiB
    T = np.full(n, 0x61, np.uint8)
    c = bw.CudaContext(n)
    try:
        src, ln = c.lz77(T)
        assert src.tolist() == [0x61, 0] and ln.tolist() == [0, n - 1]
        assert c.stats()["flags"] & bw.FLAG_LZ77
        z, outside, rounds = lz_counters(c)
        assert z == 2 and rounds == 0  # the path leaves tile 0 straight to the end
    finally:
        c.close()


# ---- tile edges -----------------------------------------------------------------------------------------------------
def _edge_sizes():
    out = set()
    for edge in (LZ_GROUP, LZ_ROW_TILE, 2 * LZ_ROW_TILE, LZ_TEXT_TILE, 2 * LZ_TEXT_TILE, 3 * LZ_TEXT_TILE):
        out |= {edge - 1, edge, edge + 1}
    return sorted(out)


@pytest.mark.parametrize("n", _edge_sizes())
def test_tile_edges(ctx, n):
    """Texts ending at and around every tile size of the new kernels, in three shapes: short phrases (binary), rows
    whose PSV / NSV leave their tile (one byte: every row), and a phrase spanning several text tiles (a repeat)."""
    rng = np.random.default_rng(n)
    for shape in ("binary", "one_byte", "repeat"):
        if shape == "binary":
            T = rng.integers(0, 2, n).astype(np.uint8)
        elif shape == "one_byte":
            T = np.full(n, 7, np.uint8)
        else:
            T = np.resize(rng.integers(0, 256, min(n, 700)).astype(np.uint8), n).astype(np.uint8)
        src, ln = with_oracle(ctx, T, (n, shape))
        z, outside, rounds = lz_counters(ctx)
        assert z == src.size
        if shape == "one_byte" and n > LZ_ROW_TILE:
            assert outside >= n - 1  # no row has a smaller SA value above it
        assert rounds <= max(0, (-(-n // LZ_TEXT_TILE) - 1).bit_length())


def test_phrase_starts_on_text_tile_boundaries(ctx):
    """Random bytes give short phrases: across many tiles, some start exactly at a multiple of LZ_TEXT_TILE."""
    T = np.random.default_rng(3).integers(0, 256, 64 * LZ_TEXT_TILE + 17).astype(np.uint8)
    src, ln = with_oracle(ctx, T, "boundaries")
    starts = np.concatenate([[0], np.cumsum(np.maximum(1, ln))[:-1]])
    assert (starts[starts > 0] % LZ_TEXT_TILE == 0).sum() >= 2
    assert lz_counters(ctx)[2] >= 1  # the marking rounds crossed tiles


# ---- the capacity contract ------------------------------------------------------------------------------------------
def test_capacity_contract(ctx):
    T = bw.generate("markov", 300000, seed=103)
    want_src, want_len = oracle_lz77(T, ctx.divsufsort(T))
    z = want_src.size
    lib, h = ctx._lib, ctx._h
    assert lib.bwtc_cuda_lz77(h, T.ctypes.data, T.size, None, None, 0) == z  # count query
    src, ln = np.full(z, -5, np.int32), np.full(z, -6, np.int32)
    assert lib.bwtc_cuda_lz77(h, T.ctypes.data, T.size, src.ctypes.data, ln.ctypes.data, z - 1) == z
    assert (src == -5).all() and (ln == -6).all()
    assert lib.bwtc_cuda_lz77(h, T.ctypes.data, T.size, src.ctypes.data, ln.ctypes.data, z) == z
    assert np.array_equal(src, want_src) and np.array_equal(ln, want_len)
    with pytest.raises(ValueError):
        ctx.lz77(T, np.zeros(z - 1, np.int32), np.zeros(z, np.int32))


# ---- buffer kinds ---------------------------------------------------------------------------------------------------
def test_host_buffer_kinds(ctx):
    """Pageable and pinned src / len in all four combinations; more than one staging-ring chunk of phrases."""
    T = np.random.default_rng(4).integers(0, 256, 6 * MiB).astype(np.uint8)
    want_src, want_len = oracle_lz77(T, ctx.divsufsort(T))
    z = want_src.size
    assert z * 4 > (4 << 20)
    _, ps = _pinned(np.zeros(z, np.int32))
    _, pl = _pinned(np.zeros(z, np.int32))
    for s, l in ((np.zeros(z, np.int32), np.zeros(z, np.int32)), (ps, np.zeros(z, np.int32)),
                 (np.zeros(z, np.int32), pl), (ps, pl)):
        s[:] = 0
        l[:] = 0
        gs, gl = ctx.lz77(T, s, l)
        assert np.array_equal(gs, want_src) and np.array_equal(gl, want_len)


def test_device_buffers(ctx):
    import torch

    T = bw.generate("dna", 2 * MiB + 3, seed=104)
    want_src, want_len = oracle_lz77(T, ctx.divsufsort(T))
    z = want_src.size
    dT = torch.from_numpy(T).cuda()
    buf = torch.full((2 * z + 8,), -1, dtype=torch.int32, device="cuda")
    d_src, d_len = buf.data_ptr(), buf.data_ptr() + 4 * (z + 4)
    assert ctx.lz77_device(dT.data_ptr(), T.size, 0, 0, 0) == z
    assert ctx.lz77_device(dT.data_ptr(), T.size, d_src, d_len, z - 1) == z
    assert (buf == -1).all().item()
    assert ctx.lz77_device(dT.data_ptr(), T.size, d_src, d_len, z) == z
    h = buf.cpu().numpy()
    assert np.array_equal(h[:z], want_src) and np.array_equal(h[z + 4:2 * z + 4], want_len)
    assert (h[z:z + 4] == -1).all() and (h[2 * z + 4:] == -1).all()
    # a text at an odd device address (unpadded): read only within its n bytes
    dT2 = torch.zeros(T.size + 1, dtype=torch.uint8, device="cuda")
    dT2[1:] = dT
    buf.fill_(-1)
    assert ctx.lz77_device(dT2.data_ptr() + 1, T.size, d_src, d_len, z) == z
    h = buf.cpu().numpy()
    assert np.array_equal(h[:z], want_src) and np.array_equal(h[z + 4:2 * z + 4], want_len)
    # n == 1 on the device
    assert ctx.lz77_device(dT2.data_ptr() + 1, 1, d_src, d_len, 1) == 1
    assert buf[0].item() == int(T[0]) and buf[z + 4].item() == 0
    # misaligned or overlapping arrays
    for a, b, cap in ((d_src + 2, d_len, z), (d_src, d_len + 1, z), (d_src, d_src + 4 * (z - 1), z), (0, d_len, z),
                      (d_src, d_src, 1)):
        with pytest.raises(bw.BwtcCudaError) as ei:
            ctx.lz77_device(dT.data_ptr(), T.size, a, b, cap)
        assert ei.value.code == EARG, (a - d_src, b - d_src, cap)
    assert ctx.lz77_device(dT.data_ptr(), T.size, d_src, d_src + 4 * z, z) == z  # adjacent, not overlapping


def test_limits_and_argument_errors():
    lib = bw.load_library()
    c = bw.CudaContext(1 << 16)
    try:
        T = np.zeros((1 << 16) + 2, np.uint8)
        s = np.zeros(T.size, np.int32)
        assert lib.bwtc_cuda_lz77(c._h, T.ctypes.data, (1 << 16) + 2, s.ctypes.data, s.ctypes.data, 0) == ETOOBIG
        assert lib.bwtc_cuda_lz77_device(c._h, T.ctypes.data, (1 << 16) + 2, None, None, 0) == ETOOBIG
        assert lib.bwtc_cuda_lz77(c._h, None, 5, None, None, 0) == EARG
        assert lib.bwtc_cuda_lz77_device(c._h, None, 5, None, None, 0) == EARG
        assert lib.bwtc_cuda_lz77(c._h, T.ctypes.data, 5, None, s.ctypes.data, 5) == EARG
        assert lib.bwtc_cuda_lz77(c._h, T.ctypes.data, 5, s.ctypes.data, None, 5) == EARG
        assert lib.bwtc_cuda_lz77(None, T.ctypes.data, 5, None, None, 0) == EARG
        # the largest text the context takes (cap + 1 bytes) still works
        T = bw.generate("markov", (1 << 16) + 1, seed=105)
        with_oracle(c, T, "cap + 1")
    finally:
        c.close()


# ---- engine paths ---------------------------------------------------------------------------------------------------
_ENGINE = {}


def _engine_cases(oracle):
    if not _ENGINE:
        for i, kind in enumerate(KINDS):
            T = bw.generate(kind, 2 * MiB + 5 + i, seed=106)
            _ENGINE[kind] = (T, oracle_lz77(T, oracle_sa(oracle, T)))
    return _ENGINE.items()


@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()) or "default")
def test_every_engine_path(oracle, monkeypatch, knobs):
    """Whatever buffers the sort's path leaves behind, the LCP and LZ77 stages read the SA and the text correctly."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    tickets = knobs.get("BWTC_STATIC_TILES") == "0" or knobs.get("BWTC_DEBUG_FAKE_WATCHDOG") == "1"
    c = bw.CudaContext(4 * MiB)
    try:
        for kind, (T, (want_src, want_len)) in _engine_cases(oracle):
            check(c, T, want_src, want_len, (kind, knobs))
            assert bool(c.stats()["flags"] & F_TICKETS) == tickets, kind
    finally:
        c.close()


# ---- verification, flags, stats and leakage -------------------------------------------------------------------------
def test_verified_results_are_unchanged(ctx):
    T = bw.generate("repetitive", 2 * MiB + 1, seed=107)
    want = ctx.lz77(T)
    want = (want[0].copy(), want[1].copy())
    ctx.set_verify(True)
    try:
        src, ln = ctx.lz77(T)
        fl = ctx.stats()["flags"]
        assert fl & bw.FLAG_VERIFIED and fl & bw.FLAG_SA and fl & bw.FLAG_LCP and fl & bw.FLAG_LZ77
        assert np.array_equal(src, want[0]) and np.array_equal(ln, want[1])
    finally:
        ctx.set_verify(False)


@pytest.mark.parametrize("row", ["0", "last"])
def test_corrupt_sa_hook_gives_everify(monkeypatch, row):
    """BWTC_DEBUG_CORRUPT_SA=r: EVERIFY, and pageable / pinned / device src and len keep their previous contents."""
    import torch

    T = bw.generate("markov", MiB + 11, seed=108)
    n = T.size
    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_SA", str(n - 2) if row == "last" else row)
    c = bw.CudaContext(2 * MiB)
    try:
        c.set_verify(True)
        _, pS = _pinned(np.full(n, 123, np.int32))
        _, pL = _pinned(np.full(n, 321, np.int32))
        for S, L in ((np.full(n, 123, np.int32), np.full(n, 321, np.int32)), (pS, pL)):
            with pytest.raises(bw.BwtcCudaError) as ei:
                c.lz77(T, S, L)
            assert ei.value.code == bw.EVERIFY
            assert (S == 123).all() and (L == 321).all()
        dT = torch.from_numpy(T).cuda()
        d = torch.full((2 * n,), 5, dtype=torch.int32, device="cuda")
        with pytest.raises(bw.BwtcCudaError) as ei:
            c.lz77_device(dT.data_ptr(), n, d.data_ptr(), d.data_ptr() + 4 * n, n)
        assert ei.value.code == bw.EVERIFY and (d == 5).all().item()
        c.set_verify(False)
        src, ln = c.lz77(T)
        assert np.array_equal(decode(src, ln, n), T)
    finally:
        c.close()


def test_stats_record():
    T = bw.generate("markov", 3 * MiB + 1, seed=109)
    c = bw.CudaContext(4 * MiB)
    try:
        c.divsufsort_lcp(T)
        lcp_st = c.stats()
        src, ln = c.lz77(T)
        st = c.stats()
        assert st["n_suffixes"] == T.size
        assert st["flags"] & (bw.FLAG_SA | bw.FLAG_LCP | bw.FLAG_LZ77) == bw.FLAG_SA | bw.FLAG_LCP | bw.FLAG_LZ77
        assert not st["flags"] & bw.FLAG_VERIFIED and not lcp_st["flags"] & bw.FLAG_LZ77
        assert st["kernel_launches"] > lcp_st["kernel_launches"]
        assert st["algorithmic_bytes"] > lcp_st["algorithmic_bytes"] and st["gpu_ms"] > 0
        z, outside, rounds = lz_counters(c)
        assert z == src.size and 0 < outside < T.size
        assert 1 <= rounds <= (-(-T.size // LZ_TEXT_TILE) - 1).bit_length()
        # debug_read(9) still holds the LCP stage's counters: the same as after divsufsort_lcp
        irr = c.debug_read(9, np.uint64, 1)[0]
        c.divsufsort_lcp(T)
        assert c.debug_read(9, np.uint64, 1)[0] == irr
    finally:
        c.close()


def test_watchdog_retry_gives_the_same_phrases(oracle, monkeypatch):
    T = bw.generate("repetitive", 3 * MiB, seed=110)
    want = oracle_lz77(T, oracle_sa(oracle, T))
    monkeypatch.setenv("BWTC_DEBUG_FAKE_WATCHDOG", "1")
    c = bw.CudaContext(4 * MiB)
    try:
        check(c, T, *want, "watchdog")
        assert c.stats()["flags"] & F_TICKETS
    finally:
        c.close()


def _other_calls(c, T, x):
    """divsufsort_lcp, sa_search and divbwtf: results, launch counts and flags."""
    SA, LCP = c.divsufsort_lcp(T)
    out = [("divsufsort_lcp", SA.copy(), LCP.copy())]
    st = c.stats()
    out.append(("divsufsort_lcp stats", st["kernel_launches"], st["flags"]))
    P, P_off = bw.pack_patterns([T[i:i + k].tobytes() for i, k in ((0, 5), (1000, 40), (77, 3))] + [b"zz"])
    left, size = c.sa_search(T, SA, P, P_off)
    out.append(("sa_search", left.copy(), size.copy()))
    U = np.zeros(x.size, np.uint8)
    LF = np.zeros(256, np.uint32)
    fr = np.zeros(256, np.uint32)
    out.append(("divbwtf", c.divbwtf(x, U, LF, fr), U.copy(), LF.copy(), fr.copy()))
    st = c.stats()
    out.append(("divbwtf stats", st["kernel_launches"], st["flags"]))
    return out


def test_flags_and_no_leakage():
    """Around lz77 calls on one context, divsufsort_lcp, sa_search and divbwtf give a fresh context's results, launch
    counts and flags (bit 12 clear); lz77 gives the same phrases between them; scratch_bytes is unchanged."""
    T = bw.generate("markov", MiB + 3, seed=111)
    x = bw.generate("dna", 300000, seed=112)
    cap = 2 * MiB
    scratch = bw.load_library().bwtc_cuda_scratch_bytes(cap)
    fresh = bw.CudaContext(cap)
    try:
        want = _other_calls(fresh, T, x)
        ws, wl = fresh.lz77(T)
        ws, wl = ws.copy(), wl.copy()
    finally:
        fresh.close()
    for g in want:
        if g[0].endswith("stats"):
            assert not g[2] & bw.FLAG_LZ77, g
    c = bw.CudaContext(cap)
    try:
        for _ in range(2):
            src, ln = c.lz77(T)
            assert np.array_equal(src, ws) and np.array_equal(ln, wl)
            got = _other_calls(c, T, x)
            for p, q in zip(got, want):
                assert p[0] == q[0]
                for u, v in zip(p[1:], q[1:]):
                    assert np.array_equal(u, v) if isinstance(u, np.ndarray) else u == v, (p[0], u, v)
        assert bw.load_library().bwtc_cuda_scratch_bytes(cap) == scratch
        assert np.array_equal(decode(ws, wl, T.size), T)
    finally:
        c.close()
