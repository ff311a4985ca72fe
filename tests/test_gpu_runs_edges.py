"""GPU tests of the run statistics (bwtc_cuda_bwt_block_runs, bwtc_cuda_pipeline_submit_runs; k_run_count / k_run_emit in
ibwt_kernels.cuh, queued behind k_finish in every ladder chunk of phase_sort) at the edges where they can go wrong: the
16-byte thread and 4096-byte tile boundaries of run_heads16 and its scalar tail, the sweeps of k_scan_tile_counts (16384
tiles each, a carried prefix), the capacity contract, errors, every engine path, buffer kinds, the look-back status rows
the tile counts borrow, and the pipeline's grouping rule that keeps a runs block out of a batch.

The C ABI is called through ctypes with caller-owned run arrays filled with sentinels, so that a write past `count`, or
any write on overflow or on an error, is seen.  The reference for the runs is always a numpy scan of the output bytes,
heads = {0} u {i : out[i] != out[i-1]}; the output bytes themselves are checked against the C oracle (up to ~2 MiB), the
recorded oracle digests (full-size generated blocks), or bwtc_cuda_bwt_block of the same input on a fresh context."""
import ctypes

import numpy as np
import pytest

import bwtc_b200 as bw
from conftest import digest
from test_gpu_parity import ENGINE_KNOBS

pytestmark = pytest.mark.gpu

GUARD = 0x5A
SYM_SENT, START_SENT = 0xA5, 0xDEADBEEF
LF_SENT, FR0 = 0x77777777, 3
OVERFLOW = bw.RUNS_OVERFLOW
EARG, ETOOBIG = -1, -5
F_TICKETS = 1
TILE, SWEEP = 4096, 4096 * 16384  # RUN_TILE; tiles per k_scan_tile_counts sweep (1024 threads x 16)


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _lib():
    return bw.load_library()


def _pin(a):
    import torch

    return torch.from_numpy(a).pin_memory().numpy()


class Call:
    """One bwtc_cuda_bwt_block_runs call: the block in a buffer with a guard byte behind it, LFpowers and freqs filled
    with sentinels, run arrays of `slots` entries filled with sentinels (NULL where asked)."""

    def __init__(self, ctx, x, capacity, slots=None, pinned_block=False, pinned_runs=False, null_sym=False,
                 null_start=False, count0=12345, block_ptr=True, n=None):
        n = x.size if n is None else n
        self.x = x
        buf = np.empty(x.size + 1, np.uint8)
        buf[:-1] = x
        buf[-1] = GUARD
        self.buf = _pin(buf) if pinned_block else buf
        self.out = self.buf[:-1]
        self.LF = np.full(bw.num_starting_points(max(n, 1), 8), LF_SENT, np.uint32)
        self.fr = np.full(256, FR0, np.uint32)
        if slots is None:
            slots = min(capacity, x.size) + 8
        sym = np.full(slots, SYM_SENT, np.uint8)
        start = np.full(slots, START_SENT, np.uint32)
        self.sym, self.start = (_pin(sym), _pin(start)) if pinned_runs else (sym, start)
        self.r = bw.Runs(capacity, count0, None if null_sym else self.sym.ctypes.data,
                         None if null_start else self.start.ctypes.data)
        h = ctx._h if ctx is not None else None
        self.rc = _lib().bwtc_cuda_bwt_block_runs(h, self.buf.ctypes.data if block_ptr else None, n, self.LF.ctypes.data,
                                                  self.LF.size, self.fr.ctypes.data, ctypes.addressof(self.r))
        self.count = self.r.count

    def check_block(self, want):
        """The block contract's outputs against want = (out, LF, freqs), the guard byte, pidx."""
        assert self.rc >= 0, self.rc
        assert self.buf[-1] == GUARD, "the byte after the block was written"
        assert self.rc == self.LF[0]
        assert np.array_equal(self.LF, want[1]), "LFpowers"
        assert np.array_equal(self.fr - FR0, want[2]), "freqs"
        assert np.array_equal(self.out, want[0]), ("BWT bytes", int(np.count_nonzero(self.out != want[0])))

    def check_runs(self):
        check_runs(self.out, self.count, self.sym, self.start)

    def check_untouched_runs(self):
        assert self.count == OVERFLOW, self.count
        assert (self.sym == SYM_SENT).all() and (self.start == START_SENT).all(), "run arrays written on overflow / error"

    def check_untouched_inputs(self):
        assert np.array_equal(self.out, self.x) and self.buf[-1] == GUARD, "block written"
        assert (self.LF == LF_SENT).all() and (self.fr == FR0).all(), "LFpowers / freqs written"


def count_runs(out):
    return 1 + int(np.count_nonzero(out[1:] != out[:-1])) if out.size else 0


def check_runs(out, count, sym, start, chunk=16 << 20):
    """count / symbol / start equal a scan of out (chunked: bounded host memory at 256 MiB); every entry from `count` on
    still holds its sentinel."""
    n = out.size
    assert count != OVERFLOW, "overflow reported where the runs fit"
    off = 0
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        m = np.empty(b - a, bool)
        m[0] = a == 0 or out[a] != out[a - 1]
        m[1:] = out[a + 1:b] != out[a:b - 1]
        h = np.flatnonzero(m).astype(np.uint32) + np.uint32(a)
        k = h.size
        assert off + k <= count, ("more runs than reported", count)
        assert np.array_equal(start[off:off + k], h), ("start", a)
        assert np.array_equal(sym[off:off + k], out[h]), ("symbol", a)
        off += k
    assert off == count, (off, count)
    assert (sym[count:] == SYM_SENT).all() and (start[count:] == START_SENT).all(), "run arrays written past count"


def boundary_kinds(out):
    """Which head decisions at thread (16j, not a tile start) and tile (4096j) starts this output exercises.  A kernel that
    took prev = 0 at a thread start fails on 'equal_nonzero' (a head where there is none) and 'zero_after_nonzero' (a head
    missed)."""
    n = out.size
    kinds = set()
    for level, step in (("thread", 16), ("tile", TILE)):
        j = np.arange(step, n, step)
        if level == "thread":
            j = j[j % TILE != 0]
        if j.size == 0:
            continue
        cur, prev = out[j], out[j - 1]
        if np.any((cur == prev) & (cur != 0)):
            kinds.add((level, "equal_nonzero"))
        if np.any((cur == 0) & (prev != 0)):
            kinds.add((level, "zero_after_nonzero"))
    return kinds


def fresh_block(x, cap=None):
    """bwtc_cuda_bwt_block of x on a fresh context: (out, LF, freqs, kernel_launches)."""
    ctx = bw.CudaContext(cap or x.size)
    try:
        out = x.copy()
        LF = np.zeros(bw.num_starting_points(x.size, 8), np.uint32)
        fr = np.zeros(256, np.uint32)
        ctx.bwt_block(out, LF, fr)
        return out, LF, fr, ctx.stats()["kernel_launches"]
    finally:
        ctx.close()


_ORACLE = {}


def oracle_of(oracle, key, x):
    if key not in _ORACLE:
        _ORACLE[key] = oracle.block(x, 8)
    return _ORACLE[key]


def edge_inputs(n, rng):
    """Random inputs at sigma = 2, 3, 256, and outputs built to carry runs across 16- and 4096-byte boundaries."""
    k = max(1, n // 2)
    yield "zeros", np.zeros(n, np.uint8)
    yield "sigma2", rng.integers(0, 2, n).astype(np.uint8)
    yield "sigma3", rng.integers(0, 3, n).astype(np.uint8)
    yield "sigma256", rng.integers(0, 256, n).astype(np.uint8)
    yield "abab", np.resize(np.array([0x61, 0x62], np.uint8), n)
    yield "aabb", np.concatenate([np.full(k, 0x61, np.uint8), np.full(n - k, 0x62, np.uint8)])
    yield "00ff", (rng.integers(0, 2, n) * 0xFF).astype(np.uint8)
    yield "descending", (np.arange(n, 0, -1) % 251 + 1).astype(np.uint8)


# ---- 1. thread and tile edges ------------------------------------------------------------------------------------------
EDGE_SIZES = (list(range(1, 41)) + [TILE * k + d for k in (1, 2, 3) for d in (-1, 0, 1)]
              + [16 * m + r for m in (4095, 4096) for r in range(16)])


def test_runs_at_thread_and_tile_edges(oracle):
    """Every size 1..40 (the scalar tail of run_heads16 only), 4096k - 1 / 4096k / 4096k + 1, and 16m + r around 64 KiB
    (every tail length 0..15 behind full 16-byte groups).  The outputs must put zero and non-zero bytes on both sides of
    thread and tile starts, and the filled hole byte at pidx = 1, n - 1 and n (pidx is never 0 in the block contract)."""
    rng = np.random.default_rng(101)
    ctx = bw.CudaContext(max(EDGE_SIZES))
    kinds, pidx_kinds = set(), set()
    try:
        for n in EDGE_SIZES:
            for name, x in edge_inputs(n, rng):
                want = oracle.block(x, 8)
                c = Call(ctx, x, capacity=n)
                c.check_block(want)
                c.check_runs()
                kinds |= boundary_kinds(c.out)
                p = int(c.rc)
                pidx_kinds.add("1" if p == 1 else "n-1" if p == n - 1 else "n" if p == n else "mid")
    finally:
        ctx.close()
    assert kinds == {(lv, k) for lv in ("thread", "tile") for k in ("equal_nonzero", "zero_after_nonzero")}, kinds
    assert {"1", "n-1", "n", "mid"} <= pidx_kinds, pidx_kinds


# ---- 2. sweep edges of the tile scan ----------------------------------------------------------------------------------
def _runs_full(x, capacity, want=None, record=None):
    n = x.size
    ctx = bw.CudaContext(n)
    try:
        c = Call(ctx, x, capacity=capacity, slots=n + 8)
    finally:
        ctx.close()
    if record is not None:
        assert c.rc >= 0 and c.buf[-1] == GUARD
        record.check(x, 8, c.out, c.LF, c.fr - FR0)
    else:
        c.check_block(want)
    c.check_runs()
    return c


def test_runs_one_full_sweep_of_tiles(oracle_record):
    """64 MiB of DNA: exactly 16384 tiles, one full sweep of k_scan_tile_counts, no carry used."""
    x = bw.generate("dna", 64 << 20, seed=31)
    assert -(-x.size // TILE) == 16384
    _runs_full(x, x.size, record=oracle_record)


@pytest.mark.parametrize("extra", [1, TILE + 1])
def test_runs_past_the_first_sweep(extra):
    """64 MiB + 1 and + 4097 bytes: 16385 and 16386 tiles, the first blocks whose run offsets (and the total) need the
    prefix carried into the second sweep."""
    x = bw.generate("dna", SWEEP + extra, seed=33)
    want = fresh_block(x)
    c = _runs_full(x, x.size, want=want[:3])
    assert -(-x.size // TILE) == 16384 + (1 if extra == 1 else 2)
    assert c.count > 1


def test_runs_of_256mib_random_block(oracle_record):
    """65536 tiles (4 sweeps), about 2.7e8 runs, capacity = n: the run arrays take 1.3 GB of host memory."""
    x = bw.generate("random", 256 << 20, seed=31)
    c = _runs_full(x, x.size, record=oracle_record)
    assert c.count > (250 << 20)


def test_runs_of_96mib_repetitive_block():
    """A large repetitive block with few runs (what the compressor ships): a fresh context's bwt_block is the reference."""
    x = bw.generate("repetitive", 96 << 20, seed=34)
    want = fresh_block(x)
    c = _runs_full(x, x.size // 8, want=want[:3])
    assert c.count <= x.size // 8


# ---- 3. capacity contract ---------------------------------------------------------------------------------------------
def test_capacity_contract(oracle):
    """Capacity 0, 1, count - 1, count, count + 1, n, n + 1 and 0xFFFFFFFF; NULL arrays; runs = NULL.  On overflow every
    sentinel survives, on success every entry from `count` on; the block is transformed either way.  A runs call costs
    three run-kernel launches per ladder chunk and 2n algorithmic bytes more than the same bwt_block call."""
    n = (1 << 20) + 3
    x = bw.generate("repetitive", n, seed=61)
    want = oracle.block(x, 8)
    cnt = count_runs(want[0])
    assert 1 < cnt < n
    ctx = bw.CudaContext(n)
    try:
        for cap in (0, 1, cnt - 1, cnt, cnt + 1, n, n + 1, 0xFFFFFFFF):
            c = Call(ctx, x, capacity=cap, slots=min(cap, n + 1) + 8)
            c.check_block(want)
            if cap < cnt:
                c.check_untouched_runs()
            else:
                c.check_runs()
        for null_sym, null_start in ((True, False), (False, True), (True, True)):
            c = Call(ctx, x, capacity=n, null_sym=null_sym, null_start=null_start)
            c.check_block(want)
            c.check_untouched_runs()
        # runs = NULL is bwt_block, launch for launch
        blk = x.copy()
        LF = np.zeros(bw.num_starting_points(n, 8), np.uint32)
        fr = np.zeros(256, np.uint32)
        rc = _lib().bwtc_cuda_bwt_block_runs(ctx._h, blk.ctypes.data, n, LF.ctypes.data, LF.size, fr.ctypes.data, None)
        st_null = ctx.stats()
        assert rc == want[1][0] and np.array_equal(blk, want[0]) and np.array_equal(LF, want[1])
        blk = x.copy()
        ctx.bwt_block(blk, LF, None)
        st_plain = ctx.stats()
        assert st_null["kernel_launches"] == st_plain["kernel_launches"]
        assert st_null["algorithmic_bytes"] == st_plain["algorithmic_bytes"]
        Call(ctx, x, capacity=n).check_runs()
        st_runs = ctx.stats()
        # the run kernels are queued behind k_finish in every ladder chunk (3 launches each), their bytes count once
        extra = st_runs["kernel_launches"] - st_plain["kernel_launches"]
        assert extra >= 3 and extra % 3 == 0, extra
        assert st_runs["algorithmic_bytes"] == st_plain["algorithmic_bytes"] + 2 * n
    finally:
        ctx.close()


# ---- 4. errors --------------------------------------------------------------------------------------------------------
def test_argument_errors_report_overflow(oracle):
    """Null block, n == 0, a null context, a block above the capacity: count = BWTC_CUDA_RUNS_OVERFLOW, the run arrays,
    block, LFpowers and freqs untouched, the context still usable."""
    n = 4096
    x = bw.generate("markov", n + 1, seed=62)
    ctx = bw.CudaContext(n)
    try:
        for kw in ({"block_ptr": False, "n": n}, {"n": 0}):
            c = Call(ctx, x[:n], capacity=n, **kw)
            assert c.rc == EARG, c.rc
            c.check_untouched_runs()
            c.check_untouched_inputs()
        c = Call(None, x[:n], capacity=n)
        assert c.rc == EARG
        c.check_untouched_runs()
        c.check_untouched_inputs()
        c = Call(ctx, x, capacity=n + 1)
        assert c.rc == ETOOBIG, c.rc
        c.check_untouched_runs()
        c.check_untouched_inputs()
        c = Call(ctx, x[:n], capacity=n)
        c.check_block(oracle.block(x[:n], 8))
        c.check_runs()
    finally:
        ctx.close()


def test_everify_reports_overflow(oracle, monkeypatch):
    """With verification on and a corrupted output (test hook), the call fails with EVERIFY after the runs were
    downloaded: count must still read overflow; block, LFpowers and freqs hold their inputs (the run arrays are
    unspecified).  The context stays usable."""
    monkeypatch.setenv("BWTC_DEBUG_CORRUPT_OUT", "1")
    n = 100003
    ctx = bw.CudaContext(n)
    monkeypatch.delenv("BWTC_DEBUG_CORRUPT_OUT")
    try:
        ctx.set_verify(True)
        x = bw.generate("repetitive", n, seed=63)
        for pinned in (False, True):
            c = Call(ctx, x, capacity=n, pinned_block=pinned)
            assert c.rc == bw.EVERIFY, c.rc
            assert c.count == OVERFLOW, c.count
            if not pinned:
                c.check_untouched_inputs()
            assert (c.LF == LF_SENT).all() and (c.fr == FR0).all()
        ctx.set_verify(False)
        c = Call(ctx, x, capacity=n)
        c.check_block(oracle.block(x, 8))
        c.check_runs()
    finally:
        ctx.close()


def test_unfinished_block_reports_overflow(oracle):
    """set_debug(max_rounds) stops the block unfinished: its runs were never computed, so the call reports overflow and
    leaves the arrays alone (not a count of 0)."""
    n = 100003
    x = bw.generate("markov", n, seed=64)
    ctx = bw.CudaContext(n)
    try:
        ctx.set_debug(1)
        c = Call(ctx, x, capacity=n)
        assert c.rc >= 0
        c.check_untouched_runs()
        ctx.set_debug(0)
        c = Call(ctx, x, capacity=n)
        c.check_block(oracle.block(x, 8))
        c.check_runs()
    finally:
        ctx.close()


# ---- 5. every engine path ---------------------------------------------------------------------------------------------
KNOB_N = (2 << 20) + 4097


@pytest.mark.parametrize("knobs", ENGINE_KNOBS, ids=lambda k: ",".join(f"{a[5:]}={b}" for a, b in k.items()) or "default")
def test_every_engine_path_runs(oracle, monkeypatch, knobs):
    """Every knob setting of test_gpu_parity on Markov, DNA, repetitive (multi-chunk ladders, global radix rounds) and
    random blocks: exact bytes and exact runs."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    ctx = bw.CudaContext(KNOB_N)
    tickets = knobs.get("BWTC_STATIC_TILES") == "0" or knobs.get("BWTC_DEBUG_FAKE_WATCHDOG") == "1"
    try:
        for kind in ("markov", "dna", "repetitive", "random"):
            x = bw.generate(kind, KNOB_N, seed=65)
            c = Call(ctx, x, capacity=KNOB_N)
            c.check_block(oracle_of(oracle, kind, x))
            c.check_runs()
            st = ctx.stats()
            assert bool(st["flags"] & F_TICKETS) == tickets, (kind, st["flags"])
            if kind == "repetitive" and not knobs:
                assert st["rounds"] > 2 and max(st["passes"][1:st["rounds"]]) > 0, "expected global radix rounds"
    finally:
        ctx.close()


@pytest.mark.parametrize("force", [(1, 4), (3, 4), (2, 8), (5, 8), (64, 8)])
def test_runs_with_forced_round0_key_shapes(oracle, force):
    rng = np.random.default_rng(66)
    ctx = bw.CudaContext(70001)
    ctx.set_round0(*force)
    try:
        for n in (1, 17, 4097, 70001):
            for name, x in edge_inputs(n, rng):
                if name in ("sigma256", "descending") and n > 4097:
                    continue
                c = Call(ctx, x, capacity=n)
                c.check_block(oracle.block(x, 8))
                c.check_runs()
    finally:
        ctx.close()


def test_runs_with_verification(oracle):
    ctx = bw.CudaContext(KNOB_N)
    ctx.set_verify(True)
    try:
        for kind in ("markov", "repetitive"):
            x = bw.generate(kind, KNOB_N, seed=65)
            c = Call(ctx, x, capacity=KNOB_N)
            c.check_block(oracle_of(oracle, kind, x))
            c.check_runs()
            assert ctx.stats()["flags"] & bw.FLAG_VERIFIED
    finally:
        ctx.close()


def test_runs_after_a_watchdog_retry(oracle, monkeypatch):
    """The fake watchdog fails the first attempt after the run kernels ran; the retry with tickets must give exact runs."""
    monkeypatch.setenv("BWTC_DEBUG_FAKE_WATCHDOG", "1")
    ctx = bw.CudaContext(KNOB_N)
    monkeypatch.delenv("BWTC_DEBUG_FAKE_WATCHDOG")
    try:
        x = bw.generate("repetitive", KNOB_N, seed=65)
        c = Call(ctx, x, capacity=KNOB_N)
        c.check_block(oracle_of(oracle, "repetitive", x))
        c.check_runs()
        assert ctx.stats()["flags"] & F_TICKETS
    finally:
        ctx.close()


# ---- 6. buffer kinds --------------------------------------------------------------------------------------------------
def test_buffer_kinds(oracle):
    """Pageable and pinned blocks, pageable and pinned run arrays (the start array of ~1.6 M runs is larger than one 4 MiB
    chunk of the staging ring), and calls with different capacities on one context."""
    x = bw.generate("markov", KNOB_N, seed=65)
    want = oracle_of(oracle, "markov", x)
    cnt = count_runs(want[0])
    assert cnt * 4 > (4 << 20)
    ctx = bw.CudaContext(KNOB_N)
    try:
        for pb in (False, True):
            for pr in (False, True):
                c = Call(ctx, x, capacity=KNOB_N, pinned_block=pb, pinned_runs=pr)
                c.check_block(want)
                c.check_runs()
        for cap in (cnt, cnt - 1, KNOB_N // 8, KNOB_N, cnt):
            c = Call(ctx, x, capacity=cap)
            c.check_block(want)
            if cap < cnt:
                c.check_untouched_runs()
            else:
                c.check_runs()
    finally:
        ctx.close()


# ---- 7. context reuse after a runs call -------------------------------------------------------------------------------
REUSE_CAP = 16 << 20


def _ops(oracle):
    """(name, fn(ctx) -> comparable result) of every other entry point, on inputs smaller than the runs block."""
    xb = bw.generate("markov", (1 << 20) + 3, seed=67)
    xs = [bw.generate("markov", 1 << 17, seed=68 + i) for i in range(8)]
    xi = bw.generate("dna", 300001, seed=69)
    fwd_i = oracle.block(xi, 8)
    T = bw.generate("random", 300001, seed=70)
    xr = bw.generate("repetitive", 100003, seed=71)

    def block(ctx):
        b = xb.copy()
        LF = np.zeros(8, np.uint32)
        fr = np.zeros(256, np.uint32)
        p = ctx.bwt_block(b, LF, fr)
        return p, digest(b), LF.tolist(), fr.tolist()

    def blocks(ctx):
        bl = [x.copy() for x in xs]
        LF, nLF, fr = ctx.bwt_blocks(bl, 8)
        return [digest(b) for b in bl], LF.tolist(), nLF.tolist(), fr.tolist()

    def inverse(ctx):
        b = fwd_i[0].copy()
        ctx.inverse_block(b, fwd_i[1])
        assert np.array_equal(b, xi)
        return digest(b)

    def divbwtf(ctx):
        U = np.zeros_like(T)  # (U[pidx] is left as it was)
        LF = np.zeros(8, np.uint32)
        fr = np.zeros(256, np.uint32)
        p = ctx.divbwtf(T, U, LF, fr)
        return p, digest(U), LF.tolist(), fr.tolist()

    def divsufsort(ctx):
        return digest(ctx.divsufsort(T))

    def runs(ctx):
        c = Call(ctx, xr, capacity=xr.size)
        c.check_runs()
        return c.rc, digest(c.out), c.count, digest(c.sym), digest(c.start)

    return [("bwt_block", block), ("bwt_blocks", blocks), ("inverse_block", inverse), ("divbwtf", divbwtf),
            ("divsufsort", divsufsort), ("runs", runs)]


def test_context_reuse_around_a_runs_call(oracle, oracle_record):
    """The tile counts of a runs call live in the pass-0 look-back status rows.  After the runs of a 16 MiB repetitive
    block (4096 tiles of counts and offsets in those rows), every other entry point on the same context must give what a
    fresh context gives, with the same kernel launches; and a runs call after each of them must too."""
    ops = _ops(oracle)
    want = {}
    for name, fn in ops:
        ctx = bw.CudaContext(REUSE_CAP)
        try:
            want[name] = (fn(ctx), ctx.stats()["kernel_launches"])
        finally:
            ctx.close()
    big = bw.generate("repetitive", REUSE_CAP, seed=31)
    run_fn = dict(ops)["runs"]
    ctx = bw.CudaContext(REUSE_CAP)
    try:
        for name, fn in ops:
            c = Call(ctx, big, capacity=REUSE_CAP)
            assert c.rc >= 0
            oracle_record.check(big, 8, c.out, c.LF, c.fr - FR0)
            c.check_runs()
            got = (fn(ctx), ctx.stats()["kernel_launches"])
            assert got == want[name], name
            got = (run_fn(ctx), ctx.stats()["kernel_launches"])
            assert got == want["runs"], ("runs after", name)
    finally:
        ctx.close()


# ---- pipeline ---------------------------------------------------------------------------------------------------------
PIPE_N = 1 << 16


def _plain_inputs(oracle, count=16):
    return [(x, oracle_of(oracle, ("pipe", i), x)) for i, x in
            ((i, bw.generate("markov", PIPE_N, seed=200 + i)) for i in range(count))]


def _check_runs_result(res, want):
    LF, fr, runs = res
    out = want[0]
    assert np.array_equal(LF, want[1]) and np.array_equal(fr, want[2])
    assert runs is not None, "runs not filled (was the block batched?)"
    sym, start = runs
    h = np.flatnonzero(np.concatenate([[True], out[1:] != out[:-1]]))
    assert np.array_equal(start, h) and np.array_equal(sym, out[h])


def test_pipeline_runs_block_behind_a_batch(oracle):
    """8 equal small plain blocks, a small runs block of the same size, 8 more plain blocks, all queued before the first
    wait, depth 1, several times.  The worker takes the first block alone and then groups what has queued up behind it:
    the runs block must end that group.  Exact runs prove it was transformed on its own (the batch path never fills
    runs, count would stay overflow).  The grouping is timing-dependent; the assertions are not."""
    plain = _plain_inputs(oracle)
    xr = bw.generate("repetitive", PIPE_N, seed=210)
    wr = oracle.block(xr, 8)
    p = bw.Pipeline(PIPE_N, depth=1)
    try:
        for rep in range(6):
            blocks = [x.copy() for x, _ in plain]
            hs = [p.submit(b, 8) for b in blocks[:8]]
            rb = xr.copy()
            hr = p.submit_runs(rb, PIPE_N)
            hs += [p.submit(b, 8) for b in blocks[8:]]
            for (x, w), b, h in zip(plain, blocks, hs):
                LF, fr = p.wait(h)
                assert np.array_equal(b, w[0]) and np.array_equal(LF, w[1]) and np.array_equal(fr, w[2]), rep
            _check_runs_result(p.wait(hr), wr)
            assert np.array_equal(rb, wr[0])
    finally:
        p.close()


@pytest.mark.parametrize("depth", [1, 2, 4])
@pytest.mark.parametrize("verify", [False, True])
def test_pipeline_runs_mixed_and_out_of_place(oracle, depth, verify):
    """Several runs blocks in flight (in place and out of place: `in` stays unchanged), between plain forward blocks and
    inverse items, with and without verification."""
    plain = _plain_inputs(oracle, 6)
    xs = [bw.generate(k, PIPE_N - 7 * i, seed=220 + i) for i, k in enumerate(["repetitive", "markov", "dna", "repetitive"])]
    ws = [oracle.block(x, 8) for x in xs]
    p = bw.Pipeline(PIPE_N, depth=depth)
    p.set_verify(verify)
    try:
        items = []
        for i, (x, w) in enumerate(zip(xs, ws)):
            src = x.copy()
            dst = np.full(x.size, 0xEE, np.uint8) if i % 2 else None
            items.append(("runs", p.submit_runs(src, x.size, out=dst), (x, w, src, dst)))
            px, pw = plain[i]
            b = px.copy()
            items.append(("plain", p.submit(b, 8), (b, pw)))
            ib = pw[0].copy()
            items.append(("inverse", p.submit_inverse(ib, pw[1]), (ib, px)))
        for kind, h, data in items:
            r = p.wait(h)
            if kind == "runs":
                x, w, src, dst = data
                _check_runs_result(r, w)
                if dst is None:
                    assert np.array_equal(src, w[0])
                else:
                    assert np.array_equal(src, x), "out-of-place input was written"
                    assert np.array_equal(dst, w[0])
            elif kind == "plain":
                b, w = data
                assert np.array_equal(b, w[0]) and np.array_equal(r[0], w[1]) and np.array_equal(r[1], w[2])
            else:
                ib, px = data
                assert np.array_equal(ib, px)
    finally:
        p.close()


def test_pipeline_runs_ticket_error_reports_overflow():
    """A runs block above the contexts' capacity fails its ticket with ETOOBIG and leaves count = overflow; the pipeline
    goes on."""
    p = bw.Pipeline(PIPE_N, depth=1)  # contexts hold a batch: 64 blocks of PIPE_N bytes
    try:
        x = bw.generate("markov", 64 * PIPE_N + 65, seed=230)
        h = p.submit_runs(x.copy(), 1000)
        with pytest.raises(bw.BwtcCudaError) as ei:
            p.wait(h)
        assert ei.value.code == ETOOBIG
        assert h["runs"].count == OVERFLOW
        assert (h["sym"] == 0).all() and (h["start"] == 0).all()
        y = bw.generate("repetitive", PIPE_N, seed=231)
        b = y.copy()
        res = p.wait(p.submit_runs(b, PIPE_N))
        assert res[2] is not None and res[2][0].size == count_runs(b)
    finally:
        p.close()
