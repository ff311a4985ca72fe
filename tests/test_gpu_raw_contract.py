"""GPU tests of the RAW forward contract, bwtc_cuda_divbwt / bwtc_cuda_divbwtf (divsufsort.h:86-94): the path a bwtc build
runs through the link-time divsufsort shim and through CudaBWTransform::doTransform(byte*, ...), which get
T = reverse(X)·0x00 of |X| + 1 bytes from the reference's BWTransform::doTransform(BWTBlock&).  The raw contract is never
verified at run time (DESIGN.md §3.10), and it runs code the block contract does not: the last byte always joins the
alphabet (DNA gets 3-bit codes and the gram projection, Markov text a 65th symbol), the text is read from the unpadded,
reused input buffer, `out[pidx] = text[pidx]` on the device and a result copy in two ranges around pidx on the host.

Every case compares all four outputs (U, the returned pidx, LFpowers, freqs), most from a buffer with a guard byte behind
U.  References: the C oracle's raw transform, or — at full block size, where the oracle's outputs are recorded for the
block contract only — the block contract's recorded result, from which the raw result of T = reverse(X)·0x00 follows
exactly (raw_from_block, checked against the oracle on the CPU)."""
import math

import numpy as np
import pytest

import bwtc_b200 as bw
from test_gpu_parity import ENGINE_KNOBS

GUARD = 0x5A
F_TICKETS, F_PACKED, F_AUX, F_LAZY = 1, 4, 8, 16
RING_CHUNK = 4 << 20  # bwt_engine.cu: chunk of the pinned staging ring that pageable results are copied through
ETOOBIG = -5


def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


def gpu(test):
    return pytest.mark.gpu(pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")(test))


# ---- references and the engine's rules, restated ---------------------------------------------------------------------
def raw_text(x):
    """T = reverse(X)·0x00: what BWTransform::doTransform(BWTBlock&) hands to the raw contract."""
    T = np.empty(x.size + 1, np.uint8)
    T[:-1] = x[::-1]
    T[-1] = 0
    return T


def raw_from_block(T, out, p):
    """The raw contract's in-place U for T = reverse(X)·0x00 (N = n + 1 bytes), from the block contract's output `out`
    (n bytes) and pidx p.  Both hold L = BWT(T) in rows r != p, r < n; the block contract moves L[N-1] into the hole at p,
    the raw contract leaves U[p] = T[p] and keeps L[N-1] in row n.  p == n: row n is the hole itself and keeps T[n] = 0.
    LFpowers and freqs are the same for both contracts."""
    n = out.size
    U = np.append(out, T[n])
    if p < n:
        U[n] = out[p]
        U[p] = T[p]
    return U


def _ceil_log2(v):
    return (int(v) - 1).bit_length()


def _code_bits(sigma):
    return 1 if sigma <= 2 else _ceil_log2(sigma)


def raw_alphabet(T):
    """(sigma, bits per character) of a raw text: every byte of T, the last one included, is a character."""
    sigma = int(np.count_nonzero(np.bincount(T, minlength=256)))
    return sigma, _code_bits(sigma)


def policy_flags(T, st, iid):
    """stats flags 4 / 8 / 16 plan_round0, round0 and choose_lazy choose at default knobs: the predecessor code packed above the id
    when both fit 32 bits, else a one-byte payload from 96 Mi suffixes on; lazy ranks for an i.i.d. source (no memory)
    whose predicted live fraction after round 0, 1 - exp(-N 2^(-H0 c)), is at most 0.065, from 4 Mi suffixes on."""
    N = T.size
    packed = max(1, _ceil_log2(N)) + st["bits_per_char"] <= 32
    aux = not packed and N >= (96 << 20)
    cnt = np.bincount(T, minlength=256).astype(np.float64)
    q = cnt[cnt > 0] / N
    H0 = float(-(q * np.log2(q)).sum())
    live = 1.0 - math.exp(-N * 2.0 ** (-H0 * st["chars_round0"]))
    lazy = iid and live <= 0.065 and N >= (4 << 20)
    return (F_PACKED if packed else 0) | (F_AUX if aux else 0) | (F_LAZY if lazy else 0)


def run_raw(ctx, T, nLF, out=None, fr0=0):
    """divbwtf(T, U, ...) with U = T in place (out None) or U = a copy of `out`; U sits in a buffer with a guard byte.
    Returns (pidx, U, LFpowers, freqs)."""
    buf = np.empty(T.size + 1, np.uint8)
    buf[:-1] = T if out is None else out
    buf[-1] = GUARD
    U = buf[:-1]
    LF = np.zeros(nLF, np.uint32)
    fr = np.full(256, fr0, np.uint32)
    pidx = ctx.divbwtf(U if out is None else T, U, LF, fr)
    assert buf[-1] == GUARD, "the byte after U was written"
    return pidx, U, LF, fr


def assert_raw(got, want, what):
    pidx, U, LF, fr = got
    rc, wU, wLF, wfr = want
    assert pidx == rc == wLF[0] == LF[0], ("pidx", what, pidx, rc)
    assert np.array_equal(LF, wLF), ("LFpowers", what)
    assert (fr is None and wfr is None) or np.array_equal(fr, wfr), ("freqs", what)
    assert np.array_equal(U, wU), ("U", what, int(np.count_nonzero(U != wU)))


# ---- the derivation from the block contract, on the CPU ---------------------------------------------------------------
def test_raw_from_block_matches_the_oracle(oracle):
    """raw_from_block(T, block output, pidx) equals the oracle's raw transform of T = reverse(X)·0x00, LFpowers and freqs
    equal the block contract's; among the blocks, ones whose pidx is n (suffix 0 of T sorts last) and 1 (first after
    the terminator's suffix)."""
    rng = np.random.default_rng(90)
    blocks = [np.full(n, 7, np.uint8) for n in (1, 2, 3, 300)]  # reverse(X)·0x00 = 7...7 0: suffix 0 is the largest
    blocks += [np.arange(n, 0, -1).astype(np.uint8) for n in (2, 200)]  # descending X: T ascending, pidx = 1
    blocks += [rng.integers(0, s, n).astype(np.uint8) for n in (1, 2, 5, 257, 1000, 4099) for s in (1, 2, 4, 256)]
    seen = set()
    for x in blocks:
        n = x.size
        out, LF, fr = oracle.block(x, 8)
        T = raw_text(x)
        rc, wU, wLF, wfr = oracle.raw(T, LF.size)
        p = int(LF[0])
        seen.add("n" if p == n else ("1" if p == 1 else "mid"))
        assert rc == p and np.array_equal(wLF, LF) and np.array_equal(wfr, fr), n
        assert np.array_equal(raw_from_block(T, out, p), wU), (n, p)
    assert seen == {"n", "1", "mid"}, seen


# ---- 1. full block size: raw and block contract compute the same transform ------------------------------------------
@gpu
@pytest.mark.parametrize("kind,mib", [("markov", 32), ("dna", 64), ("repetitive", 16), ("random", 256)])
def test_full_size_raw_equals_recorded_block_result(oracle_record, kind, mib):
    """The BASELINE block sizes of test_gpu_fullsize.py: the block contract's result is checked against the recorded oracle
    digests, the raw call on T = reverse(X)·0x00 must give exactly the result derived from it.  stats() shows the raw run's
    own alphabet (DNA: A, C, G, T and the terminator = 3-bit codes, the gram path; Markov: 65 symbols) and flags."""
    x = bw.generate(kind, mib << 20, seed=31)
    n = x.size
    ctx = bw.CudaContext(n + 1)
    try:
        blk = x.copy()
        LF = np.zeros(bw.num_starting_points(n, 8), np.uint32)
        fr = np.zeros(256, np.uint32)
        p = ctx.bwt_block(blk, LF, fr)
        oracle_record.check(x, 8, blk, LF, fr)
        T = raw_text(x)
        del x
        want = (p, raw_from_block(T, blk, p), LF, fr)
        del blk
        got = run_raw(ctx, T, LF.size)
        st = ctx.stats()
    finally:
        ctx.close()
    assert_raw(got, want, kind)
    sigma, bits = raw_alphabet(T)
    assert st["n_suffixes"] == n + 1 and st["live"][0] == n + 1
    assert (st["sigma"], st["bits_per_char"]) == (sigma, bits)
    assert {"markov": (65, 7), "dna": (5, 3), "repetitive": (256, 8), "random": (256, 8)}[kind] == (sigma, bits)
    want_flags = policy_flags(T, st, iid=kind in ("dna", "random"))
    assert st["flags"] & (F_PACKED | F_AUX | F_LAZY) == want_flags, (st["flags"], want_flags)
    assert not st["flags"] & F_TICKETS


# ---- 2. every engine path, with an arbitrary last byte ---------------------------------------------------------------
N_ENGINE = (2 << 20) + 4097  # test_every_engine_path_is_bit_exact's size: 2 and 8 rank-scatter windows under its knobs
KINDS = ("markov", "dna", "repetitive", "random")
LAST_BYTE_FORMS = ("zero_absent", "zero_inside", "largest", "unique", "tail_run")


def last_byte_form(R, form, rng):
    """A raw text from the body R (N - 1 bytes, modified in place) and one form of its last byte:
    zero_absent  0x00 that occurs nowhere else (what integration options A and B send);
    zero_inside  0x00 that also occurs inside the text;
    largest      the largest byte value of the text;
    unique       a value between the smallest and the largest that occurs nowhere else;
    tail_run     the smallest value, ending a run of 3000: windows running past the end (code-0 padding) tie with real
                 code-0 characters."""
    if form == "zero_absent":
        np.maximum(R, 1, out=R)
        last = 0
    elif form == "zero_inside":
        R[rng.integers(0, R.size, 1000)] = 0
        last = 0
    elif form == "largest":
        last = int(R.max())
    elif form == "unique":
        last = (int(R.min()) + int(R.max())) // 2
        R[R == last] = last + 1
    else:
        last = int(R.min())
        R[-2999:] = last
    return np.append(R, np.uint8(last))


_ENGINE_CASES = []


def engine_cases(oracle):
    """(name, T, oracle raw result with 8 LFpowers) for every family x last-byte form, computed once per module."""
    if not _ENGINE_CASES:
        rng = np.random.default_rng(91)
        for kind in KINDS:
            for form in LAST_BYTE_FORMS:
                R = np.ascontiguousarray(bw.generate(kind, N_ENGINE - 1, seed=43)[::-1])
                T = last_byte_form(R, form, rng)
                _ENGINE_CASES.append((f"{kind}/{form}", T, oracle.raw(T, 8)))
    return _ENGINE_CASES


@gpu
@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()) or "default")
def test_every_engine_path_raw(oracle, monkeypatch, knobs):
    """The knob settings of test_every_engine_path_is_bit_exact on raw texts of about 2 MiB: four families x five forms of
    the last byte, all the oracle's outputs.  Tile tickets and lazy ranks as the knobs demand, for every call."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    tickets = knobs.get("BWTC_STATIC_TILES") == "0" or knobs.get("BWTC_DEBUG_FAKE_WATCHDOG") == "1"
    cases = engine_cases(oracle)
    ctx = bw.CudaContext(N_ENGINE)
    try:
        for name, T, want in cases:
            assert_raw(run_raw(ctx, T, 8), want, (name, knobs))
            st = ctx.stats()
            assert (st["sigma"], st["bits_per_char"]) == raw_alphabet(T), name
            assert bool(st["flags"] & F_TICKETS) == tickets, (name, st["flags"])
            if knobs.get("BWTC_LAZY") == "2":
                assert st["flags"] & F_LAZY, (name, "lazy ranks should have been used")
    finally:
        ctx.close()


def _small_raw_texts(rng):
    """Raw texts from 2 bytes to 150 KB over 1, 2, 4 and 200 symbols, each with four last bytes: the smallest symbol (a
    tail run of it for longer texts), the largest, a unique value and 0x00."""
    for n in (2, 3, 5, 17, 40, 63, 64, 65, 100, 1000, 150001):
        for sigma in (1, 2, 4, 200):
            body = (rng.integers(0, sigma, n - 1) + 30).astype(np.uint8)
            for last in ("min", "max", "unique", "zero"):
                R = body.copy()
                if last == "min":
                    v = int(R.min()) if R.size else 30
                    R[-min(R.size, 50):] = v
                elif last == "max":
                    v = int(R.max()) if R.size else 30
                elif last == "unique":
                    v = 29 if n % 2 else 255
                else:
                    v = 0
                yield f"n={n},sigma={sigma},last={last}", np.append(R, np.uint8(v))


@gpu
@pytest.mark.parametrize("force", [(0, 0), (1, 4), (3, 4), (2, 8), (5, 8), (64, 8)])
def test_raw_forced_round0_key_shapes(oracle, force):
    """Forced round-0 key shapes on raw texts, including windows longer than the whole text (64 one-bit characters on a
    40-byte text: short_thresh = 0, every window runs past the end)."""
    rng = np.random.default_rng(92)
    ctx = bw.CudaContext(150001)
    ctx.set_round0(*force)
    try:
        for name, T in _small_raw_texts(rng):
            nLF = min(T.size, 8)
            assert_raw(run_raw(ctx, T, nLF), oracle.raw(T, nLF), (name, force))
    finally:
        ctx.close()


@gpu
@pytest.mark.parametrize("gram", ["1", "0"])
@pytest.mark.parametrize("sigma,force", [(8, (0, 0)), (8, (4, 4)), (8, (10, 4)), (8, (21, 8)), (64, (2, 4)), (64, (3, 4)),
                                         (64, (10, 8))])
def test_raw_gram_projection(oracle, monkeypatch, gram, sigma, force):
    """3- and 6-bit raw alphabets with BWTC_GRAM=1 (digit histograms projected from one gram histogram) and 0, where the
    last byte makes the alphabet: sigma - 1 data values plus a unique smallest / largest last byte, or sigma data values
    ending in a run of the largest."""
    monkeypatch.setenv("BWTC_GRAM", gram)
    rng = np.random.default_rng(2000 + sigma)
    for n, form in ((70001, "unique_min"), (300007, "max_run"), (65, "unique_max")):
        if form == "max_run":
            R = rng.integers(0, sigma, n - 1).astype(np.uint8)
            R[:sigma] = np.arange(sigma, dtype=np.uint8)
            R[-30:] = sigma - 1
            T = np.append(R, np.uint8(sigma - 1))
        else:
            R = (rng.integers(0, sigma - 1, n - 1) + (1 if form == "unique_min" else 0)).astype(np.uint8)
            R[: sigma - 1] = np.arange(sigma - 1, dtype=np.uint8) + (1 if form == "unique_min" else 0)
            T = np.append(R, np.uint8(0 if form == "unique_min" else 200))
        c = bw.CudaContext(n)
        c.set_round0(*force)
        try:
            got = run_raw(c, T, 8)
            st = c.stats()
        finally:
            c.close()
        assert_raw(got, oracle.raw(T, 8), (n, form))
        assert (st["sigma"], st["bits_per_char"]) == (sigma, _code_bits(sigma)), (n, form)


# ---- 3. the host copy of the result around pidx -----------------------------------------------------------------------
N_COPY = 2 * RING_CHUNK + 4099
PLACEMENTS = [0, 1, RING_CHUNK - 1, RING_CHUNK, RING_CHUNK + 1, 2 * RING_CHUNK, N_COPY - 2, N_COPY - 1]


def text_with_pidx(p, rng):
    """N_COPY random bytes with T[0] = 0x80 occurring nowhere else and exactly p smaller bytes: suffix 0 then has rank
    #{i : T[i] < T[0]} = p."""
    rest = np.concatenate([rng.integers(0, 0x80, p), rng.integers(0x81, 0x100, N_COPY - 1 - p)]).astype(np.uint8)
    rng.shuffle(rest)
    return np.concatenate([np.array([0x80], np.uint8), rest])


def _pinned(n):
    import torch

    return torch.empty(n, dtype=torch.uint8).pin_memory()


@pytest.fixture(scope="module")
def copy_ctx():
    c = bw.CudaContext(N_COPY)
    yield c
    c.close()


@gpu
@pytest.mark.parametrize("p", PLACEMENTS)
def test_pidx_at_the_edges_of_the_result_copy(oracle, copy_ctx, p):
    """The result reaches the caller in two ranges around pidx: two cudaMemcpyAsync into a pinned U, chunks of the 4 MiB
    staging ring into a pageable one.  pidx at 0, 1, a ring chunk +-1, two chunks, n - 2 and n - 1; pageable and pinned
    buffers, in place and into a separate U filled with a marker that U[pidx] must keep.  (The device-side output holds
    T[pidx] there, different from the marker: a copy that includes row pidx shows.)"""
    rng = np.random.default_rng(93 + p)
    T = text_with_pidx(p, rng)
    rc, wU, wLF, wfr = oracle.raw(T, 8)
    assert rc == p
    marker = 0x80 if p else 0xEE  # never T[p]
    keep = np.ones(N_COPY, bool)
    keep[p] = False
    hold = []
    for pinned in (False, True):
        for separate in (False, True):
            if pinned:
                tb, ub = _pinned(N_COPY + 1), _pinned(N_COPY + 1)
                hold += [tb, ub]
                tbuf, ubuf = tb.numpy(), ub.numpy()
            else:
                tbuf, ubuf = np.empty(N_COPY + 1, np.uint8), np.empty(N_COPY + 1, np.uint8)
            tbuf[:-1] = T
            tbuf[-1] = GUARD
            ubuf[:-1] = marker
            ubuf[-1] = GUARD
            src = tbuf[:-1]
            U = ubuf[:-1] if separate else src
            LF = np.zeros(8, np.uint32)
            fr = np.zeros(256, np.uint32)
            what = (p, "pinned" if pinned else "pageable", "separate" if separate else "in place")
            assert copy_ctx.divbwtf(src, U, LF, fr) == p, what
            assert tbuf[-1] == GUARD and ubuf[-1] == GUARD, what
            assert np.array_equal(LF, wLF) and np.array_equal(fr, wfr), what
            assert U[p] == (marker if separate else T[p]), (what, "U[pidx] must stay untouched", int(U[p]))
            assert np.array_equal(U[keep], wU[keep]), (what, int(np.count_nonzero(U[keep] != wU[keep])))
            if separate:
                assert np.array_equal(src, T), (what, "T was written")


# ---- 4. contract edges ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(1 << 20)
    yield c
    c.close()


@gpu
def test_divbwt_and_divbwtf_without_freqs(ctx, oracle):
    """bwtc_cuda_divbwt (no freqs argument: what CudaBWTransform::doTransform(byte*, uint32, LF) calls) through ctypes, and
    divbwtf with freqs = NULL, both in place and into a separate U."""
    lib = bw.load_library()
    rng = np.random.default_rng(94)
    for n, sigma in ((2, 2), (1000, 4), (70001, 256), (300000, 64)):
        T = rng.integers(0, sigma, n).astype(np.uint8)
        T[-1] = 0
        nLF = min(n, 8)
        rc, wU, wLF, _ = oracle.raw(T, nLF)
        for separate in (False, True):
            buf = np.full(n + 1, GUARD, np.uint8)
            buf[:-1] = 0xEE if separate else T
            src = T.copy() if separate else buf[:-1]
            LF = np.zeros(nLF, np.uint32)
            got = lib.bwtc_cuda_divbwt(ctx._h, src.ctypes.data, buf.ctypes.data, n, LF.ctypes.data, nLF)
            assert got == rc and np.array_equal(LF, wLF) and buf[-1] == GUARD, (n, separate)
            keep = np.arange(n) != rc
            assert np.array_equal(buf[:-1][keep], wU[keep]) and buf[rc] == (0xEE if separate else T[rc]), (n, separate)
        U = T.copy()
        LF = np.zeros(nLF, np.uint32)
        assert_raw((ctx.divbwtf(U, U, LF, None), U, LF, None), (rc, wU, wLF, None), ("divbwtf, freqs NULL", n))


@gpu
def test_trivial_sizes_return_early(ctx, oracle):
    """n = 0 and n = 1 never reach the sort (divsufsort.c:488-489): n is returned, U[0] = T[0] for n = 1, LFpowers and
    freqs stay untouched — through divbwtf and divbwt."""
    lib = bw.load_library()
    for n in (0, 1):
        T = np.array([9, GUARD], np.uint8)
        U = np.array([0xEE, GUARD], np.uint8)
        LF = np.array([77], np.uint32)
        fr = np.full(256, 5, np.uint32)
        assert ctx._check(lib.bwtc_cuda_divbwtf(ctx._h, T.ctypes.data, U.ctypes.data, n, LF.ctypes.data, 1, fr.ctypes.data)) == n
        assert U[0] == (9 if n else 0xEE) and U[1] == GUARD and T[0] == 9 and LF[0] == 77 and (fr == 5).all(), n
        U[0] = 0xEE
        assert lib.bwtc_cuda_divbwt(ctx._h, T.ctypes.data, U.ctypes.data, n, LF.ctypes.data, 1) == n
        assert U[0] == (9 if n else 0xEE) and LF[0] == 77, n
    rc, buf, wLF, wfr = oracle.raw(np.array([9], np.uint8), 1)
    assert rc == 1 and buf[0] == 9 and wfr.sum() == 0


@gpu
def test_one_lfpower_per_suffix(ctx, oracle):
    """nLF = N gives x = N / nLF = 1: every suffix N - j is sampled.  256 LFpowers at N = 256 and N = 257 (x = 1 too), N = 2,
    on texts with and without T[N-2] < T[N-1].  There the reference's divsufsort never samples suffix N - 1 and leaves
    LFpowers[1] as it was (DESIGN.md §1); the engine returns its true rank, taken here from the suffix array."""
    rng = np.random.default_rng(95)
    quirks = 0
    for N, nLF in ((256, 256), (257, 256), (2, 2), (3, 3), (300, 256)):
        for sigma in (2, 4, 256):
            for order in ("up", "down", "any"):
                T = rng.integers(0, sigma, N).astype(np.uint8)
                if order != "any" and T[-2] == T[-1]:
                    T[-1] = T[-2] ^ 1
                if (order == "up") != (T[-2] < T[-1]) and order != "any":
                    T[-2], T[-1] = T[-1], T[-2]
                want = oracle.raw(T, nLF)
                got = run_raw(ctx, T, nLF, fr0=0)
                assert_raw(got, want, (N, nLF, sigma, order))
                if N // nLF == 1 and T[N - 2] < T[N - 1]:
                    _, ISA = oracle.suffix_array(T)
                    assert got[2][1] == ISA[N - 1], (N, sigma, "LFpowers[1] must be the rank of suffix N - 1")
                    quirks += 1
    assert quirks >= 6


@gpu
def test_errors_leave_every_buffer_untouched(oracle):
    """nLF > N (x would be 0) returns EARG; a raw text longer than capacity + 1 returns ETOOBIG.  Neither writes U,
    LFpowers or freqs."""
    c = bw.CudaContext(1000)
    try:
        for n, nLF, code in ((4, 8, -1), (100, 101, -1), (1002, 8, ETOOBIG), (5000, 8, ETOOBIG)):
            T = np.random.default_rng(n).integers(0, 4, n).astype(np.uint8)
            for separate in (False, True):
                U = np.full(n, 0xEE, np.uint8) if separate else T.copy()
                src = T.copy() if separate else U
                LF = np.full(nLF, 77, np.uint32)
                fr = np.full(256, 5, np.uint32)
                with pytest.raises(bw.BwtcCudaError) as e:
                    c.divbwtf(src, U, LF, fr)
                assert e.value.code == code, (n, nLF, e.value)
                assert (U == (0xEE if separate else T)).all() and (LF == 77).all() and (fr == 5).all(), (n, nLF, separate)
        # the context is still usable
        T = np.append(np.random.default_rng(1).integers(1, 9, 999), 0).astype(np.uint8)
        assert_raw(run_raw(c, T, 8), oracle.raw(T, 8), "after errors")
    finally:
        c.close()


@gpu
def test_stale_input_after_a_larger_text(oracle):
    """The raw text is read from the context's input buffer, which has no zero padding and still holds the previous call's
    bytes behind the text: a short raw call right after a large one gives exactly what it gives on a fresh context."""
    rng = np.random.default_rng(96)
    big = np.append(rng.integers(0, 256, (1 << 20) - 1), 255).astype(np.uint8)
    smalls = [T for _, T in _small_raw_texts(rng) if T.size <= 1000]
    ctx = bw.CudaContext(1 << 20)
    fresh = bw.CudaContext(1000)
    try:
        for T in smalls:
            run_raw(ctx, big, 8)
            nLF = min(T.size, 8)
            got = run_raw(ctx, T, nLF)
            assert_raw(got, oracle.raw(T, nLF), T.size)
            got_fresh = run_raw(fresh, T, nLF)
            assert all(np.array_equal(a, b) for a, b in zip(got[1:], got_fresh[1:])) and got[0] == got_fresh[0], T.size
    finally:
        ctx.close()
        fresh.close()


@gpu
def test_watchdog_retry_in_raw_mode(monkeypatch):
    """The setup of test_real_out_of_order_tiles_trip_the_watchdog_and_recover on a raw call: reversed tile order trips the
    look-back watchdog, the sort phase is repeated with tickets from the raw text still on the device.  The result equals
    the one derived from the block contract of a fresh ticket-mode context; freqs are incremented exactly once."""
    monkeypatch.setenv("BWTC_DEBUG_REVERSE_TILES", "1")
    monkeypatch.setenv("BWTC_DEBUG_SPIN_LIMIT", "2000")
    n = 12 << 20
    x = bw.generate("markov", n, seed=53)
    T = raw_text(x)
    ctx = bw.CudaContext(n + 1)
    try:
        got = run_raw(ctx, T, 8, fr0=3)
        assert ctx.stats()["flags"] & F_TICKETS, "the watchdog should have fired and the sort been repeated with tickets"
    finally:
        ctx.close()
    monkeypatch.setenv("BWTC_DEBUG_REVERSE_TILES", "0")
    monkeypatch.setenv("BWTC_STATIC_TILES", "0")
    ref = bw.CudaContext(n + 1)
    try:
        blk = x.copy()
        LF = np.zeros(8, np.uint32)
        fr = np.full(256, 3, np.uint32)
        p = ref.bwt_block(blk, LF, fr)
        assert_raw(run_raw(ref, T, 8, fr0=3), (p, raw_from_block(T, blk, p), LF, fr), "ticket context")
    finally:
        ref.close()
    assert_raw(got, (p, raw_from_block(T, blk, p), LF, fr), "after the watchdog retry")
    assert (got[3] - 3 == np.bincount(x, minlength=256)).all()


# ---- 5. capacity -------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("m", [1, 4096, 100000])
def test_capacity_is_one_more_raw_byte_than_block_bytes(oracle, m):
    """A context for blocks of m bytes holds N = m + 1 suffixes: a block of m bytes with its sentinel, or a raw text of
    m + 1 bytes (what the reference's BWTransform::doTransform(BWTBlock&) makes of an m-byte block).  m + 2 raw bytes and
    m + 1 block bytes are refused with ETOOBIG, leaving every buffer as it was."""
    rng = np.random.default_rng(97 + m)
    c = bw.CudaContext(m)
    try:
        x = rng.integers(0, 4, m).astype(np.uint8)
        T = raw_text(x)
        nLF = min(T.size, 8)
        assert_raw(run_raw(c, T, nLF), oracle.raw(T, nLF), ("m + 1", m))
        T[-1] = 3  # arbitrary last byte
        assert_raw(run_raw(c, T, nLF), oracle.raw(T, nLF), ("m + 1, last byte 3", m))
        T2 = np.append(T, np.uint8(0))
        U = np.full(m + 2, 0xEE, np.uint8)
        LF = np.full(nLF, 77, np.uint32)
        fr = np.full(256, 5, np.uint32)
        with pytest.raises(bw.BwtcCudaError) as e:
            c.divbwtf(T2, U, LF, fr)
        assert e.value.code == ETOOBIG and (U == 0xEE).all() and (LF == 77).all() and (fr == 5).all()
        blk = np.append(x, np.uint8(1))
        with pytest.raises(bw.BwtcCudaError) as e:
            c.bwt_block(blk, LF, fr)
        assert e.value.code == ETOOBIG and (LF == 77).all() and (fr == 5).all()
    finally:
        c.close()
