"""CPU restatement of the device-side LZ77 factorisation (DESIGN.md §3.14, bwt_kernels.cuh k_lz_*).

The greedy parse with self-reference: phrase k starts at p_k (p_0 = 0, p_{k+1} = p_k + max(1, len_k)), len_k is the longest
previous factor at p_k, and its source is SA[PSV] if l_P >= l_N else SA[NSV] (PSV / NSV: the nearest rows above / below
p_k's row with a smaller SA value); a literal carries its byte.  Here
  - oracle_lz77 (tests/lz77_oracle.c, which the GPU tests compare with) is pinned to brute force on every short text and
    on random texts: lengths, the source rule, and decoding back to T;
  - stage A (range minima over row tiles, a tile tree, group minima) and stage B (tile exits by pointer doubling, marking
    rounds in text order, marking inside each tile, compaction) are restated in numpy with the kernels' tile constants,
    and shown equal to the oracle, including rows whose PSV / NSV lies outside their tile, phrases spanning several text
    tiles and phrase starts exactly on a tile boundary."""
import atexit
import ctypes
import itertools
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import bwtc_b200 as bw
from test_lcp_keys import oracle_lcp
from test_sufcheck_keys import brute_sa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _constant(name):
    src = open(os.path.join(ROOT, "bwtc_b200", "csrc", "bwt_kernels.cuh")).read()
    return int(re.search(rf"constexpr uint32_t {name} = (\d+);", src).group(1))


LZ_ROW_TILE = _constant("LZ_ROW_TILE")
LZ_GROUP = _constant("LZ_GROUP")
LZ_TEXT_TILE = _constant("LZ_TEXT_TILE")
NONE = 0xFFFFFFFF

_ORACLE = []


def _oracle_lib():
    """tests/lz77_oracle.c, compiled once per process into a temporary directory (the tree may be read-only)."""
    if not _ORACLE:
        cc = shutil.which("gcc") or shutil.which("cc")
        assert cc, "no C compiler for tests/lz77_oracle.c"
        tmp = tempfile.mkdtemp(prefix="lz77_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "liblz77_oracle.so")
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-std=c99", "-Wall", "-o", out,
                        os.path.join(ROOT, "tests", "lz77_oracle.c")], check=True)
        lib = ctypes.CDLL(out)
        lib.oracle_lz77.restype = ctypes.c_int64
        lib.oracle_lz77.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                    ctypes.c_uint32]
        lib.oracle_lz77_decode.restype = ctypes.c_int64
        lib.oracle_lz77_decode.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                           ctypes.c_uint32]
        _ORACLE.append(lib)
    return _ORACLE[0]


def oracle_lz77(T, SA):
    """(src, len) of the sequential parse of T given its suffix array SA (int32[T.size])."""
    T = np.ascontiguousarray(T, np.uint8)
    SA = np.ascontiguousarray(SA, np.int32)
    src = np.empty(max(T.size, 1), np.int32)
    ln = np.empty(max(T.size, 1), np.int32)
    z = _oracle_lib().oracle_lz77(T.ctypes.data, T.size, SA.ctypes.data, src.ctypes.data, ln.ctypes.data, T.size)
    assert 0 <= z <= T.size
    return src[:z].copy(), ln[:z].copy()


def decode(src, ln, n):
    """The text the phrases stand for (byte-by-byte copies), or None if they are malformed."""
    src = np.ascontiguousarray(src, np.int32)
    ln = np.ascontiguousarray(ln, np.int32)
    out = np.empty(max(n, 1), np.uint8)
    got = _oracle_lib().oracle_lz77_decode(src.ctypes.data, ln.ctypes.data, src.size, out.ctypes.data, n)
    return out[:n] if got == n else None


def brute_lz77(T):
    """Greedy parse with lengths by brute force over all earlier starts, sources by the header's PSV / NSV rule."""
    b = bytes(np.asarray(T, np.uint8))
    n = len(b)
    SA = brute_sa(T)
    isa = np.empty(n, np.int64)
    isa[SA] = np.arange(n)

    def lcp(a, c):
        k = 0
        while a + k < n and c + k < n and b[a + k] == b[c + k]:
            k += 1
        return k

    src, ln, p = [], [], 0
    while p < n:
        best = max((lcp(p, j) for j in range(p)), default=0)
        r = isa[p]
        ps = next((SA[q] for q in range(r - 1, -1, -1) if SA[q] < p), None)
        ns = next((SA[q] for q in range(r + 1, n) if SA[q] < p), None)
        lp = lcp(p, ps) if ps is not None else 0
        lnn = lcp(p, ns) if ns is not None else 0
        assert max(lp, lnn) == best  # the PSV / NSV rule finds the longest previous factor
        src.append(b[p] if best == 0 else (ps if lp >= lnn else ns))
        ln.append(best)
        p += max(1, best)
    return np.array(src, np.int32), np.array(ln, np.int32)


def check_phrases(T, src, ln):
    """Every phrase is a literal of its byte or a copy from an earlier start; the phrases tile T and decode to it."""
    b = np.asarray(T, np.uint8)
    p = 0
    for s, l in zip(src.tolist(), ln.tolist()):
        if l == 0:
            assert s == b[p]
        else:
            assert 0 <= s < p and all(b[s + k] == b[p + k] for k in range(l))
        p += max(1, l)
    assert p == b.size
    assert np.array_equal(decode(src, ln, b.size), b)


# ---- numpy restatement of the kernels ------------------------------------------------------------------------------
def _tree(x, y, L):
    """Heap-ordered min tree of L leaves (padding: NONE)."""
    tx = np.full(2 * L, NONE, np.int64)
    ty = np.full(2 * L, NONE, np.int64)
    tx[L:L + len(x)] = x
    ty[L:L + len(y)] = y
    for k in range(L - 1, 0, -1):
        tx[k] = min(tx[2 * k], tx[2 * k + 1])
        ty[k] = min(ty[2 * k], ty[2 * k + 1])
    return tx.tolist(), ty.tolist()


def _find(tx, ty, L, i, p, right, m):
    """lz_tree_find: nearest leaf left (right) of i with x < p, or L; m lowered by y of every leaf strictly between."""
    k = L + i
    while k > 1:
        if right == (not (k & 1)):
            s = k + 1 if right else k - 1
            if tx[s] < p:
                while s < L:
                    near = 2 * s if right else 2 * s + 1
                    if tx[near] < p:
                        s = near
                    else:
                        m = min(m, ty[near])
                        s = near ^ 1
                return s - L, m
            m = min(m, ty[s])
        k >>= 1
    return L, m


def stage_a(T, SA, LCP, RT=LZ_ROW_TILE, G=LZ_GROUP):
    """k_lz_minima + k_lz_tree + k_lz_lpf: (len, src) per text position, and the rows that left their tile."""
    n = SA.size
    sa, lcp = SA.astype(np.int64).tolist(), LCP.astype(np.int64).tolist()
    ngroups = -(-n // G)
    grp = [(min(sa[g * G:(g + 1) * G]), min(lcp[g * G:(g + 1) * G])) for g in range(ngroups)]
    ntiles = -(-n // RT)
    L2 = 1 << (ntiles - 1).bit_length()
    topx, topy = _tree([min(sa[t * RT:(t + 1) * RT]) for t in range(ntiles)],
                       [min(lcp[t * RT:(t + 1) * RT]) for t in range(ntiles)], L2)
    lpf_len = np.zeros(n, np.int64)
    lpf_src = np.zeros(n, np.int64)
    outside = 0
    for t in range(ntiles):
        base = t * RT
        tx, ty = _tree(sa[base:base + RT], lcp[base:base + RT], RT)
        for k in range(min(RT, n - base)):
            r, p = base + k, sa[base + k]
            out = False
            j, m = _find(tx, ty, RT, k, p, False, NONE)
            lp, sp = min(lcp[r], m), 0
            if j < RT:
                sp = tx[RT + j]
            else:
                out = True
                t2, m = _find(topx, topy, L2, t, p, False, NONE)
                lp = min(lp, m)
                if t2 < L2:
                    g = t2 * (RT // G) + RT // G - 1
                    while True:
                        if g < ngroups:
                            if grp[g][0] < p:
                                q = min(g * G + G, n) - 1
                                while sa[q] >= p:
                                    lp = min(lp, lcp[q])
                                    q -= 1
                                sp = sa[q]
                                break
                            lp = min(lp, grp[g][1])
                        g -= 1
                else:
                    lp = 0
            j, ln = _find(tx, ty, RT, k, p, True, NONE)
            sn = 0
            if j < RT:
                ln, sn = min(ln, ty[RT + j]), tx[RT + j]
            else:
                out = True
                t2, m = _find(topx, topy, L2, t, p, True, NONE)
                ln = min(ln, m)
                if t2 < L2:
                    g = t2 * (RT // G)
                    while grp[g][0] >= p:
                        ln = min(ln, grp[g][1])
                        g += 1
                    q = g * G
                    while True:
                        ln = min(ln, lcp[q])
                        if sa[q] < p:
                            sn = sa[q]
                            break
                        q += 1
                else:
                    ln = 0
            lpf_len[p] = max(lp, ln)
            lpf_src[p] = T[p] if lpf_len[p] == 0 else (sp if lp >= ln else sn)
            outside += out
    return lpf_len, lpf_src, outside


def stage_b(lens, TT=LZ_TEXT_TILE):
    """k_lz_exit + k_lz_round + k_lz_mark_tile + k_lz_scan / k_lz_emit: the phrase starts in position order."""
    n = lens.size
    i = np.arange(n, dtype=np.int64)
    b1 = np.minimum((i // TT + 1) * TT, n)
    nxt = i + np.maximum(1, lens)

    def double(j):  # jump[i] = jump[jump[i]] inside the tile (from the previous array), unchanged past it
        inside = j < b1
        return np.where(inside, j[np.where(inside, j, 0)], j)

    ex = nxt.copy()
    while (ex < b1).any():
        ex = double(ex)
    mark = np.zeros(n, bool)
    mark[0] = True
    ttiles = -(-n // TT)
    R = (ttiles - 1).bit_length()
    jump, rounds = ex, 0
    for k in range(R):  # HBM rounds: mark jump[i] of every marked i, then double
        if rounds < k:
            break
        tgt = jump[mark & (jump < n)]
        if (~mark[tgt]).any():
            rounds = k + 1
        mark[tgt] = True
        jump = np.where(jump < n, jump[np.minimum(jump, n - 1)], n)
    entries = np.flatnonzero(mark)
    assert np.unique(entries // TT).size == entries.size  # at most one entry per tile
    jump = nxt.copy()
    while True:  # inside each tile, from its entry
        tgt = jump[mark & (jump < b1)]
        new = ~mark[tgt]
        mark[tgt] = True
        jump = double(jump)
        if not new.any():
            break
    counts = np.bincount(i[mark] // TT, minlength=ttiles)
    tpre = np.concatenate([[0], np.cumsum(counts)[:-1]])
    starts = np.flatnonzero(mark)
    assert np.array_equal(tpre[starts // TT] + (np.arange(starts.size) - tpre[starts // TT]), np.arange(starts.size))
    return starts, rounds


def model_lz77(T, SA, LCP, RT=LZ_ROW_TILE, G=LZ_GROUP, TT=LZ_TEXT_TILE):
    lens, srcs, outside = stage_a(np.asarray(T, np.uint8), SA, LCP, RT, G)
    starts, rounds = stage_b(lens, TT)
    return srcs[starts].astype(np.int32), lens[starts].astype(np.int32), dict(outside=outside, rounds=rounds,
                                                                             starts=starts)


# ---- the oracle against brute force ---------------------------------------------------------------------------------
@pytest.mark.parametrize("alphabet", [(0, 1, 2), (0x00, 0xFF)])
def test_oracle_every_short_text(alphabet):
    for n in range(1, 9):
        for t in itertools.product(alphabet, repeat=n):
            T = np.array(t, np.uint8)
            src, ln = oracle_lz77(T, brute_sa(T))
            want_src, want_len = brute_lz77(T)
            assert np.array_equal(ln, want_len) and np.array_equal(src, want_src), t
            check_phrases(T, src, ln)


def test_oracle_random_texts():
    rng = np.random.default_rng(5)
    for _ in range(300):
        n = int(rng.integers(1, 120))
        sigma = int(rng.choice([1, 2, 3, 4, 26, 256]))
        T = rng.integers(0, sigma, n).astype(np.uint8)
        if rng.random() < 0.3:  # repeats
            k = int(rng.integers(1, max(2, n // 2)))
            T = np.resize(T[:k], n).astype(np.uint8)
        src, ln = oracle_lz77(T, brute_sa(T))
        want_src, want_len = brute_lz77(T)
        assert np.array_equal(ln, want_len) and np.array_equal(src, want_src)
        check_phrases(T, src, ln)


def test_decoder_rejects_bad_phrases():
    assert decode(np.array([5, 0], np.int32), np.array([0, 2], np.int32), 3) is not None
    assert decode(np.array([5, 1], np.int32), np.array([0, 2], np.int32), 3) is None   # source not before its phrase
    assert decode(np.array([5, 0], np.int32), np.array([0, 3], np.int32), 3) is None   # past the end


# ---- the numpy model against the oracle -----------------------------------------------------------------------------
def _arrays(oracle, T):
    SA, _ = oracle.suffix_array(np.ascontiguousarray(T))
    SA = SA.view(np.int32)
    return SA, oracle_lcp(T, SA)


def test_model_small_tiles_random_texts(oracle):
    """Tiny tiles (RT 8, G 2, TT 8) put every edge of the kernels within reach of short texts."""
    rng = np.random.default_rng(6)
    for _ in range(200):
        n = int(rng.integers(2, 300))
        sigma = int(rng.choice([1, 2, 4, 256]))
        T = rng.integers(0, sigma, n).astype(np.uint8)
        if rng.random() < 0.3:
            T = np.resize(T[:int(rng.integers(1, n))], n).astype(np.uint8)
        SA, LCP = _arrays(oracle, T)
        for RT, G, TT in ((8, 2, 8), (16, 4, 4), (4, 4, 32)):
            src, ln, _ = model_lz77(T, SA, LCP, RT, G, TT)
            want_src, want_len = oracle_lz77(T, SA)
            assert np.array_equal(ln, want_len) and np.array_equal(src, want_src), (n, sigma, RT, G, TT)


def _texts_at_tile_scale():
    rng = np.random.default_rng(7)
    n = 3 * LZ_TEXT_TILE + 5
    yield "binary", rng.integers(0, 2, n).astype(np.uint8)
    yield "bytes", rng.integers(0, 256, n).astype(np.uint8)
    yield "markov", bw.generate("markov", n, seed=3)
    yield "one_byte", np.full(2 * LZ_ROW_TILE + 3, 0x61, np.uint8)
    base = rng.integers(0, 256, 1500).astype(np.uint8)  # one phrase longer than two text tiles
    yield "repeat", np.resize(base, 2 * LZ_TEXT_TILE + 3000).astype(np.uint8)


@pytest.mark.parametrize("name,T", list(_texts_at_tile_scale()), ids=lambda v: v if isinstance(v, str) else "")
def test_model_at_kernel_tiles(oracle, name, T):
    SA, LCP = _arrays(oracle, T)
    src, ln, info = model_lz77(T, SA, LCP)
    want_src, want_len = oracle_lz77(T, SA)
    assert np.array_equal(ln, want_len) and np.array_equal(src, want_src), name
    check_phrases(T, src, ln)
    assert info["outside"] > 0, name  # some rows resolved through the tile tree and the group minima
    starts, ends = info["starts"], info["starts"] + np.maximum(1, ln)
    if name == "repeat":
        assert ((ends - 1) // LZ_TEXT_TILE - starts // LZ_TEXT_TILE).max() >= 2  # a phrase spans several tiles
    if name == "bytes":
        assert (starts[starts > 0] % LZ_TEXT_TILE == 0).any()  # a phrase starts exactly on a tile boundary
