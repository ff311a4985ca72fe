"""GPU tests of bwtc_cuda_sa_search / _device (DESIGN.md §3.13): a batch of patterns counted and located in a suffix array
on the device.  Results are compared with oracle_sa_search (the sequential libdivsufsort-style search of
tests/sa_search_oracle.c, pinned to brute force by tests/test_sa_search_keys.py), with brute force on small cases and with
naive occurrence counts.  SAs come from oracle.suffix_array for small texts and from divsufsort_device for large ones."""
import math

import numpy as np
import pytest

import bwtc_b200 as bw
from test_gpu_divsufsort import _pinned, oracle_sa
from test_sa_search_keys import SEARCH_SHORT_BYTES, brute_batch, oracle_sa_search


def _has_device():
    try:
        return bw.load_library().bwtc_cuda_device_count() > 0
    except Exception:
        return False


pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not _has_device(), reason="needs a CUDA device")]

MiB = 1 << 20
EARG, ETOOBIG = -1, -5
KINDS = ("markov", "dna", "random", "repetitive", "one_byte")
LENGTHS = (1, 2, 3, 31, 32, 33, 4095, 4096, 4097, MiB)


@pytest.fixture(scope="module")
def ctx():
    c = bw.CudaContext(8 * MiB)
    yield c
    c.close()


def _text(kind, n, seed=1):
    if kind == "one_byte":
        return np.full(n, 0x61, np.uint8)
    return bw.generate(kind, n, seed=seed).copy()


def _sa(ctx, oracle, T):
    """oracle.suffix_array for small texts, divsufsort_device for large ones."""
    if T.size <= 4097:
        return np.ascontiguousarray(oracle_sa(oracle, T))
    import torch

    dT = torch.from_numpy(T).cuda()
    dSA = torch.empty(T.size, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.divsufsort_device(dT.data_ptr(), dSA.data_ptr(), T.size)
    return dSA.cpu().numpy()


def make_patterns(T, rng, per_kind=40, lengths=(1, 2, 5, 8, 16, 31, 32, 33, 100, 127, 128, 129, 1000, 4096)):
    """Hits (substrings), misses (a substring with one byte changed), prefixes running past the end of a suffix, patterns
    of n, n + 1 and n + 2 bytes, the empty pattern and all 256 one-byte patterns."""
    n = T.size
    B = T.tobytes()
    pats = [b""] + [bytes([c]) for c in range(256)]
    for m in lengths:
        if m > n:
            continue
        for s in rng.integers(0, n - m + 1, per_kind):
            p = bytearray(B[s:s + m])
            pats.append(bytes(p))
            p[int(rng.integers(0, m))] ^= int(rng.integers(1, 256))
            pats.append(bytes(p))
    for s in rng.integers(max(0, n - 40), n, min(n, 10)):  # a suffix, then more bytes
        pats.append(B[s:] + bytes(rng.integers(0, 256, int(rng.integers(1, 6))).astype(np.uint8)))
        pats.append(B[s:] + B[: int(rng.integers(1, 40))])
    pats += [B, B + B[:1], B + b"\x00", B + b"\xff\xff", B + B]
    return pats


def dev_search(ctx, T, SA, P, P_off, t_shift=0, p_shift=0):
    """sa_search_device on torch copies of the arrays; T and P start t_shift / p_shift bytes into their buffers."""
    import torch

    n, count = T.size, P_off.size - 1
    dT = torch.zeros(n + t_shift + 1, dtype=torch.uint8, device="cuda")
    if n:
        dT[t_shift:t_shift + n] = torch.from_numpy(T).cuda()
    dSA = torch.zeros(max(SA.size, 1), dtype=torch.int32, device="cuda")
    if SA.size:
        dSA[:SA.size] = torch.from_numpy(np.ascontiguousarray(SA)).cuda()
    dP = torch.zeros(P.size + p_shift + 1, dtype=torch.uint8, device="cuda")
    if P.size:
        dP[p_shift:p_shift + P.size] = torch.from_numpy(P).cuda()
    dO = torch.from_numpy(P_off.view(np.int64)).cuda()
    dL = torch.full((max(count, 1),), -77, dtype=torch.int32, device="cuda")
    dS = torch.full((max(count, 1),), -77, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.sa_search_device(dT.data_ptr() + t_shift, n, dSA.data_ptr(), SA.size, dP.data_ptr() + p_shift, dO.data_ptr(),
                         count, dL.data_ptr(), dS.data_ptr())
    return dL[:count].cpu().numpy(), dS[:count].cpu().numpy()


def check(ctx, T, SA, patterns, what, device=True, want=None):
    """Host and device variants against the C oracle (or `want`); returns the results."""
    P, P_off = patterns if isinstance(patterns, tuple) else bw.pack_patterns(patterns)
    if want is None:
        want = oracle_sa_search(T, SA, P, P_off)
    left, size = ctx.sa_search(T, SA, P, P_off)
    assert np.array_equal(size, want[1]), (what, np.flatnonzero(size != want[1])[:8].tolist())
    assert np.array_equal(left, want[0]), (what, np.flatnonzero(left != want[0])[:8].tolist())
    st = ctx.stats()
    assert st["flags"] == bw.FLAG_SEARCH and st["n_suffixes"] == T.size, (what, st["flags"])
    if device:
        dl, ds = dev_search(ctx, T, SA, P, P_off)
        assert np.array_equal(ds, want[1]) and np.array_equal(dl, want[0]), what
    return left, size


# ---- known answers --------------------------------------------------------------------------------------------------
def test_mississippi(ctx, oracle):
    T = np.frombuffer(b"mississippi", np.uint8).copy()
    SA = np.ascontiguousarray(oracle_sa(oracle, T))
    assert SA.tolist() == [10, 7, 4, 1, 0, 9, 8, 6, 3, 5, 2]
    pats = [b"", b"i", b"ssi", b"issi", b"ippi", b"mississippi", b"mississippix", b"x", b"\x00"]
    want = ([0, 0, 9, 2, 1, 4, 5, 11, 0], [11, 4, 2, 2, 1, 1, 0, 0, 0])
    want = (np.array(want[0], np.int32), np.array(want[1], np.int32))
    assert all(np.array_equal(a, b) for a, b in zip(brute_batch(T, SA, pats), want))
    check(ctx, T, SA, pats, "mississippi", want=want)


# ---- families and lengths -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", LENGTHS)
@pytest.mark.parametrize("kind", KINDS)
def test_families(ctx, oracle, kind, n):
    T = _text(kind, n, seed=n % 97 + 3)
    SA = _sa(ctx, oracle, T)
    rng = np.random.default_rng(n + len(kind))
    pats = make_patterns(T, rng, per_kind=40 if n < MiB else 200)
    left, size = check(ctx, T, SA, pats, (kind, n))
    if n <= 33:
        assert all(np.array_equal(a, b) for a, b in zip(brute_batch(T, SA, pats), (left, size))), (kind, n)


# ---- tier edges -----------------------------------------------------------------------------------------------------
def test_tier_edges(ctx, oracle):
    K = SEARCH_SHORT_BYTES
    rng = np.random.default_rng(5)
    for kind in ("markov", "repetitive", "one_byte"):
        T = _text(kind, 300_000, seed=9)
        SA = _sa(ctx, oracle, T)
        pats = make_patterns(T, rng, per_kind=60, lengths=(K - 1, K, K + 1, 127, 128, 129, 4096))
        check(ctx, T, SA, pats, kind)


def test_long_equal_runs(ctx, oracle):
    """Long matching patterns on the one-byte and the repetitive text: equal runs of thousands of bytes, up to the end."""
    rng = np.random.default_rng(6)
    for kind in ("one_byte", "repetitive"):
        T = _text(kind, 200_003, seed=4)
        SA = _sa(ctx, oracle, T)
        B = T.tobytes()
        pats = [B[s:s + m] for m in (1000, 4096, 20_000, 100_000) for s in rng.integers(0, T.size - m, 8)]
        pats += [B[-m:] for m in (33, 4096, 100_000)] + [B[-m:] + B[:5] for m in (33, 4096)]
        pats += [b"a" * m for m in (4095, 4096, 50_000, 200_003, 200_004, 200_010)]
        left, size = check(ctx, T, SA, pats, kind)
        if kind == "one_byte":
            for p, l, s in zip(pats, left, size):
                if set(p) <= {0x61} and p:
                    assert s == max(0, T.size - len(p) + 1) and l == (len(p) - 1 if s else T.size), len(p)


def test_mixed_tiers_in_random_order(ctx, oracle):
    T = _text("markov", 2 * MiB, seed=21)
    SA = _sa(ctx, oracle, T)
    rng = np.random.default_rng(8)
    pats = make_patterns(T, rng, per_kind=300, lengths=(4, 8, 20, 32, 33, 64, 500, 3000))
    order = rng.permutation(len(pats))
    check(ctx, T, SA, [pats[i] for i in order], "mixed")


# ---- SA shapes ------------------------------------------------------------------------------------------------------
def test_sa_shapes(ctx, oracle):
    rng = np.random.default_rng(10)
    for n in (1, 33, 4097, 300_000):
        T = _text("dna", n, seed=n)
        SA = _sa(ctx, oracle, T)
        pats = make_patterns(T, rng, per_kind=20, lengths=(1, 3, 12, 40, 200))
        check(ctx, T, np.concatenate([[n], SA]).astype(np.int32), pats, ("sentinel", n))
        for k in (2, 7, 64):
            check(ctx, T, np.ascontiguousarray(SA[::k]), pats, ("every k-th row", n, k))
        check(ctx, T, np.ascontiguousarray(SA[n // 2:n // 2 + 1]), pats, ("one row", n))
        check(ctx, T, np.array([n], np.int32), pats, ("only the sentinel", n))


# ---- full size ------------------------------------------------------------------------------------------------------
def test_full_size_markov(oracle):
    n, count = 32 * MiB, 100_000
    T = bw.generate("markov", n, seed=31)
    c = bw.CudaContext(n)
    try:
        SA = _sa(c, oracle, T)
        rng = np.random.default_rng(31)
        B = T.tobytes()
        lens = rng.choice([4, 8, 16, 32, 33, 64, 256, 1024], count)
        starts = rng.integers(0, n - 1024, count)
        pats = [bytearray(B[s:s + m]) for s, m in zip(starts, lens)]
        for p in pats[::2]:  # half of them misses
            p[len(p) // 2] ^= 0x5A
        P, P_off = bw.pack_patterns(pats)
        want = oracle_sa_search(T, SA, P, P_off)
        check(c, T, SA, (P, P_off), "markov 32 MiB", want=want)
        for i in rng.choice(count, 12, replace=False):  # naive occurrence counts
            p, occ, at = bytes(pats[i]), 0, B.find(bytes(pats[i]))
            while at >= 0:
                occ += 1
                at = B.find(p, at + 1)
            assert want[1][i] == occ, (i, len(p))
    finally:
        c.close()


# ---- buffer kinds ---------------------------------------------------------------------------------------------------
def test_buffer_kinds(ctx, oracle):
    """Host arrays pageable or pinned, all six at once and one pinned at a time; device arrays with T and P unaligned."""
    T = _text("markov", MiB + 5, seed=40)
    SA = _sa(ctx, oracle, T)
    rng = np.random.default_rng(40)
    P, P_off = bw.pack_patterns(make_patterns(T, rng, per_kind=100))
    want = oracle_sa_search(T, SA, P, P_off)
    count = P_off.size - 1
    arrays = {"T": T, "SA": SA, "P": P, "P_off": P_off, "left": np.zeros(count, np.int32), "size": np.zeros(count, np.int32)}
    for pinned in [set(arrays)] + [{k} for k in arrays]:
        keep, a = [], {}
        for k, v in arrays.items():
            if k in pinned:
                t, v = _pinned(v.view(np.int64) if v.dtype == np.uint64 else v.copy())
                v = v.view(np.uint64) if k == "P_off" else v
                keep.append(t)
            a[k] = v
        a["left"][:] = -9
        a["size"][:] = -9
        ctx.sa_search(a["T"], a["SA"], a["P"], a["P_off"], a["left"], a["size"])
        assert np.array_equal(a["left"], want[0]) and np.array_equal(a["size"], want[1]), sorted(pinned)
    for ts, ps in ((1, 3), (3, 1), (2, 2)):
        dl, ds = dev_search(ctx, T, SA, P, P_off, t_shift=ts, p_shift=ps)
        assert np.array_equal(dl, want[0]) and np.array_equal(ds, want[1]), (ts, ps)


# ---- chunking -------------------------------------------------------------------------------------------------------
def test_chunking_does_not_change_results(oracle):
    """A small context splits the batch into many chunks (by pattern bytes and by count); a large one takes it whole; one
    call per pattern; all three agree."""
    T = _text("repetitive", 4000, seed=12)
    SA = _sa(None, oracle, T)
    rng = np.random.default_rng(12)
    pats = make_patterns(T, rng, per_kind=150, lengths=(1, 7, 33, 200, 1500, 3999, 4000))
    pats += [bytes(T[s:s + 3]) for s in rng.integers(0, 3990, 6000)]  # more patterns than a small chunk holds
    order = rng.permutation(len(pats))
    pats = [pats[i] for i in order]
    P, P_off = bw.pack_patterns(pats)
    assert int(P_off[-1]) > 20 * 4 * 4001
    small, large = bw.CudaContext(3999), bw.CudaContext(8 * MiB)
    try:
        a = small.sa_search(T, SA, P, P_off)
        b = large.sa_search(T, SA, P, P_off)
        want = oracle_sa_search(T, SA, P, P_off)
        for r in (a, b):
            assert np.array_equal(r[0], want[0]) and np.array_equal(r[1], want[1])
        for i in rng.choice(len(pats), 300, replace=False):
            Pi, Oi = bw.pack_patterns([pats[i]])
            l1, s1 = small.sa_search(T, SA, Pi, Oi)
            assert (l1[0], s1[0]) == (a[0][i], a[1][i]), i
    finally:
        small.close()
        large.close()


# ---- limits and errors ----------------------------------------------------------------------------------------------
def test_arguments_and_limits(ctx, oracle):
    import torch

    lib, h = ctx._lib, ctx._h
    T = _text("dna", 5000, seed=2)
    SA = _sa(ctx, oracle, T)
    P, P_off = bw.pack_patterns([b"AC", b"GT", b"TTT"])
    L, S = np.full(3, 5, np.int32), np.full(3, 6, np.int32)
    args = [T.ctypes.data, T.size, SA.ctypes.data, SA.size, P.ctypes.data, P_off.ctypes.data, 3, L.ctypes.data, S.ctypes.data]
    for k in (0, 2, 4, 5, 7, 8):  # null pointers
        a = list(args)
        a[k] = None
        assert lib.bwtc_cuda_sa_search(h, *a) == EARG, k
    a = list(args)
    a[3] = T.size + 2  # SAsize > n + 1
    assert lib.bwtc_cuda_sa_search(h, *a) == EARG and "SAsize" in ctx.last_error()
    a = list(args)
    a[6] = 0  # count == 0 writes nothing
    assert lib.bwtc_cuda_sa_search(h, *a) == 0
    assert L.tolist() == [5] * 3 and S.tolist() == [6] * 3
    bad = P_off.copy()
    bad[2] = 1  # pattern 1 ends before it starts
    a = list(args)
    a[5] = bad.ctypes.data
    assert lib.bwtc_cuda_sa_search(h, *a) == EARG and "pattern 1 " in ctx.last_error()
    assert L.tolist() == [5] * 3 and S.tolist() == [6] * 3  # untouched
    small = bw.CudaContext(4096)
    try:  # host: n <= max_block_bytes + 1
        assert small._lib.bwtc_cuda_sa_search(small._h, *args) == ETOOBIG
        T2 = T[:4097].copy()
        SA2 = _sa(small, oracle, T2)
        check(small, T2, SA2, [b"AC", b"ACGT", b""], "n = capacity + 1")
        # device: not limited by the capacity
        dl, ds = dev_search(small, T, SA, P, P_off)
        want = oracle_sa_search(T, SA, P, P_off)
        assert np.array_equal(dl, want[0]) and np.array_equal(ds, want[1])
    finally:
        small.close()
    # device variant
    dT = torch.from_numpy(T).cuda()
    dSA = torch.from_numpy(SA).cuda()
    dP = torch.from_numpy(P).cuda()
    dO = torch.from_numpy(P_off.view(np.int64)).cuda()
    dBad = torch.from_numpy(bad.view(np.int64)).cuda()
    dL = torch.zeros(8, dtype=torch.int32, device="cuda")
    dS = torch.zeros(8, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    dargs = [dT.data_ptr(), T.size, dSA.data_ptr(), SA.size, dP.data_ptr(), dO.data_ptr(), 3, dL.data_ptr(), dS.data_ptr()]
    assert lib.bwtc_cuda_sa_search_device(h, *dargs) == 0
    for k in (0, 2, 4, 5, 7, 8):
        a = list(dargs)
        a[k] = None
        assert lib.bwtc_cuda_sa_search_device(h, *a) == EARG, k
    for k, shift in ((2, 2), (7, 1), (8, 2), (5, 4)):  # misaligned SA, left, size (4 bytes) and P_off (8 bytes)
        a = list(dargs)
        a[k] += shift
        assert lib.bwtc_cuda_sa_search_device(h, *a) == EARG and "aligned" in ctx.last_error(), k
    a = list(dargs)
    a[3] = T.size + 2
    assert lib.bwtc_cuda_sa_search_device(h, *a) == EARG
    a = list(dargs)
    a[6] = 0
    assert lib.bwtc_cuda_sa_search_device(h, *a) == 0
    a = list(dargs)
    a[5] = dBad.data_ptr()
    assert lib.bwtc_cuda_sa_search_device(h, *a) == EARG and "pattern 1 " in ctx.last_error()
    a = list(dargs)
    a[1] = 0x7FFFFFFF  # n above BWTC_CUDA_MAX_BLOCK + 1 (checked before anything is read)
    a[3] = 0
    assert lib.bwtc_cuda_sa_search_device(h, *a) == ETOOBIG
    # the context still works
    dl, ds = dev_search(ctx, T, SA, P, P_off)
    want = oracle_sa_search(T, SA, P, P_off)
    assert np.array_equal(dl, want[0]) and np.array_equal(ds, want[1])


def test_trivial_texts(ctx):
    """n == 0 and SAsize == 0: left = -1, size = 0; the empty pattern: left = 0, size = SAsize."""
    pats = [b"", b"a", b"\x00"]
    for T, SA, want in ((np.zeros(0, np.uint8), np.zeros(0, np.int32), ([-1] * 3, [0] * 3)),
                        (np.frombuffer(b"ab", np.uint8).copy(), np.zeros(0, np.int32), ([-1] * 3, [0] * 3)),
                        (np.zeros(0, np.uint8), np.zeros(1, np.int32), ([-1] * 3, [0] * 3)),
                        (np.frombuffer(b"a", np.uint8).copy(), np.array([0], np.int32), ([0, 0, 0], [1, 1, 0]))):
        w = (np.array(want[0], np.int32), np.array(want[1], np.int32))
        check(ctx, T, SA, pats, (T.tolist(), SA.tolist()), want=w)


def test_unsorted_sa_stays_in_range(ctx):
    rng = np.random.default_rng(13)
    T = _text("dna", 50_000, seed=13)
    n = T.size
    pats = make_patterns(T, rng, per_kind=30, lengths=(1, 4, 16, 40, 300))
    P, P_off = bw.pack_patterns(pats)
    perm = rng.permutation(n).astype(np.int32)
    wild = rng.integers(-2**31, 2**31 - 1, n + 1, dtype=np.int64).astype(np.int32)
    wild[::3] = rng.integers(n, n + 10, wild[::3].size)
    wild[1::3] = rng.integers(0, n, wild[1::3].size)
    for SA in (perm, wild, np.sort(wild)):
        for left, size in (ctx.sa_search(T, SA, P, P_off), dev_search(ctx, T, SA, P, P_off)):
            assert ((left >= -1) & (left <= SA.size)).all() and ((size >= 0) & (size <= SA.size)).all()


# ---- no leakage ----------------------------------------------------------------------------------------------------
def test_no_leakage_and_flags(ctx, oracle):
    T = _text("markov", MiB, seed=50)
    block = T.copy()
    LF = np.zeros(bw.num_starting_points(T.size, 8), np.uint32)

    def others():
        b = block.copy()
        pidx = ctx.bwt_block(b, LF, None)
        f1 = ctx.stats()["flags"]
        SA = ctx.divsufsort(T).copy()
        f2 = ctx.stats()["flags"]
        SA2, LCP = ctx.divsufsort_lcp(T)
        f3 = ctx.stats()["flags"]
        lcp_ctl = ctx.debug_read(9, np.uint64, 4)
        for f in (f1, f2, f3):
            assert not f & bw.FLAG_SEARCH
        return b, pidx, LF.copy(), SA, SA2.copy(), LCP.copy(), lcp_ctl

    before = others()
    SA = before[3]
    rng = np.random.default_rng(50)
    P, P_off = bw.pack_patterns(make_patterns(T, rng, per_kind=50))
    count = P_off.size - 1
    left, size = ctx.sa_search(T, SA, P, P_off)
    assert np.array_equal(ctx.debug_read(9, np.uint64, 4), before[6])  # the LCP stage's counters survive a search
    st = ctx.stats()
    assert st["flags"] == bw.FLAG_SEARCH and st["kernel_launches"] == 2 and st["gpu_ms"] > 0
    assert st["algorithmic_bytes"] >= 16 * count
    probes, nbytes = (int(v) for v in ctx.debug_read(10, np.uint64, 2))
    assert probes > 0 and nbytes > 0
    assert probes <= count * 2 * (math.ceil(math.log2(SA.size + 1)) + 1)
    after = others()
    for x, y in zip(before[:6], after[:6]):
        assert np.array_equal(np.asarray(x), np.asarray(y))
    ctx.set_verify(True)
    try:
        l2, s2 = ctx.sa_search(T, SA, P, P_off)
        st = ctx.stats()
        assert not st["flags"] & bw.FLAG_VERIFIED and st["flags"] & bw.FLAG_SEARCH
        assert np.array_equal(l2, left) and np.array_equal(s2, size)
        dl, ds = dev_search(ctx, T, SA, P, P_off)
        assert not ctx.stats()["flags"] & bw.FLAG_VERIFIED
        assert np.array_equal(dl, left) and np.array_equal(ds, size)
    finally:
        ctx.set_verify(False)
