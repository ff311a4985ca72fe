"""CPU tests of the pattern search's conventions (bwtc_cuda_sa_search, DESIGN.md §3.13, bwt_kernels.cuh k_sa_search_*).

Row r of an SA stands for the suffix T[SA[r]..n); an entry outside [0, n) stands for the empty suffix.  For pattern P of
m bytes, a row's key is T[s:s+m] (b"" for the empty suffix), and with the keys of a sorted SA
  left = the rows whose key sorts below P (the first matching row when there is one),  size = the rows whose key == P,
besides the special cases n == 0 or SAsize == 0 (left = -1, size = 0) and m == 0 (left = 0, size = SAsize).  Here that
definition is written out by brute force, oracle_sa_search (the sequential libdivsufsort-style search of
tests/sa_search_oracle.c that the GPU tests compare with) is pinned to it on every short text and pattern, with a sentinel
row and on sorted subsequences of the SA, and the kernels' word comparison (first differing byte from the XOR of two
little-endian words, stopping where the text or the pattern ends) is restated in numpy and checked byte by byte."""
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
from test_sufcheck_keys import brute_sa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EARG = -1


def _constant(name):
    src = open(os.path.join(ROOT, "bwtc_b200", "csrc", "bwt_kernels.cuh")).read()
    return int(re.search(rf"constexpr uint32_t {name} = (\d+);", src).group(1))


SEARCH_SHORT_BYTES = _constant("SEARCH_SHORT_BYTES")

_ORACLE = []


def _oracle_lib():
    """tests/sa_search_oracle.c, compiled once per process into a temporary directory (the tree may be read-only)."""
    if not _ORACLE:
        cc = shutil.which("gcc") or shutil.which("cc")
        assert cc, "no C compiler for tests/sa_search_oracle.c"
        tmp = tempfile.mkdtemp(prefix="sa_search_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libsa_search_oracle.so")
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-std=c99", "-Wall", "-o", out,
                        os.path.join(ROOT, "tests", "sa_search_oracle.c")], check=True)
        lib = ctypes.CDLL(out)
        lib.oracle_sa_search.restype = None
        lib.oracle_sa_search.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_uint32,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32,
                                         ctypes.c_void_p, ctypes.c_void_p]
        _ORACLE.append(lib)
    return _ORACLE[0]


def oracle_sa_search(T, SA, P, P_off, first=0, count=None, left=None, size=None):
    """(left, size) of patterns first .. first + count - 1 by the C oracle (ctypes releases the GIL: callers may run
    slices of one batch on several threads, each with its own output slices)."""
    T = np.ascontiguousarray(T, np.uint8)
    SA = np.ascontiguousarray(SA, np.int32)
    P = np.ascontiguousarray(P, np.uint8)
    P_off = np.ascontiguousarray(P_off, np.uint64)
    if count is None:
        count = P_off.size - 1 - first
    if left is None:
        left = np.empty(count, np.int32)
    if size is None:
        size = np.empty(count, np.int32)
    _oracle_lib().oracle_sa_search(T.ctypes.data, T.size, SA.ctypes.data, SA.size, P.ctypes.data, P_off.ctypes.data,
                                   first, count, left.ctypes.data, size.ctypes.data)
    return left, size


def brute_search(T, SA, pattern):
    """(left, size) of one pattern by the definition above."""
    B = bytes(np.asarray(T, np.uint8))
    n, SA = len(B), [int(s) for s in np.asarray(SA)]
    P = bytes(pattern)
    if n == 0 or not SA:
        return -1, 0
    if not P:
        return 0, len(SA)
    keys = [B[s:s + len(P)] if 0 <= s < n else b"" for s in SA]
    eq = [r for r, k in enumerate(keys) if k == P]
    if eq:
        return eq[0], len(eq)
    return sum(k < P for k in keys), 0


def brute_batch(T, SA, patterns):
    res = [brute_search(T, SA, p) for p in patterns]
    return (np.array([r[0] for r in res], np.int32), np.array([r[1] for r in res], np.int32))


def _check_oracle(T, SA, patterns, what):
    P, P_off = bw.pack_patterns(patterns)
    left, size = oracle_sa_search(T, SA, P, P_off)
    want_left, want_size = brute_batch(T, SA, patterns)
    assert np.array_equal(size, want_size), (what, size, want_size)
    assert np.array_equal(left, want_left), (what, left, want_left)


# ---- the C oracle against brute force -------------------------------------------------------------------------------
@pytest.mark.parametrize("alphabet", [(0, 1, 2), (0x00, 0xFF)])
def test_oracle_every_short_text_and_pattern(alphabet):
    patterns = [bytes(p) for m in range(5) for p in itertools.product(alphabet, repeat=m)]
    for n in range(8):
        for t in itertools.product(alphabet, repeat=n):
            T = np.array(t, np.uint8)
            SA = brute_sa(T)
            _check_oracle(T, SA, patterns, t)
            if n:  # the sentinel row: the empty suffix n first
                _check_oracle(T, np.concatenate([[n], SA]).astype(np.int32), patterns, ("sentinel", t))


def test_oracle_special_cases():
    T = np.frombuffer(b"abracadabra", np.uint8)
    SA = brute_sa(T)
    _check_oracle(T, SA, [b"", b"a", b"abra" * 4, b"abracadabra", b"abracadabrab", b"abracadabra" + b"\0" * 9], "long")
    _check_oracle(np.zeros(0, np.uint8), np.zeros(0, np.int32), [b"", b"a"], "n = 0")
    _check_oracle(T, np.zeros(0, np.int32), [b"", b"a"], "SAsize = 0")
    _check_oracle(T, np.array([11], np.int32), [b"", b"a", b"\0"], "only the empty suffix")
    _check_oracle(T, np.array([-5, 11, 99], np.int32), [b"", b"a"], "entries outside [0, n)")


def test_oracle_sorted_subsequences():
    rng = np.random.default_rng(7)
    for trial in range(60):
        n = int(rng.integers(1, 300))
        sigma = int(rng.choice([2, 3, 4, 256]))
        T = rng.integers(0, sigma, n).astype(np.uint8)
        SA = brute_sa(T)
        pats = []
        for _ in range(40):
            m = int(rng.integers(0, 12))
            s = int(rng.integers(0, n))
            p = bytearray(bytes(T[s:s + m]))
            if p and rng.random() < 0.4:
                p[int(rng.integers(0, len(p)))] = int(rng.integers(0, sigma))
            pats.append(bytes(p))
        pats += [bytes([c]) for c in range(min(sigma, 256))]
        for keep in (1.0, 0.5, 0.1):
            sub = SA[np.sort(rng.choice(n, max(1, int(n * keep)), replace=False))]
            _check_oracle(T, sub, pats, (trial, keep))
        step = int(rng.integers(2, 6))
        _check_oracle(T, SA[::step], pats, (trial, "every k-th row"))


def test_pack_patterns():
    P, P_off = bw.pack_patterns([b"ab", "", np.array([0, 255], np.uint8), "\xff"])
    assert P.dtype == np.uint8 and P_off.dtype == np.uint64
    assert P.tolist() == [97, 98, 0, 255, 255] and P_off.tolist() == [0, 2, 2, 4, 5]
    P, P_off = bw.pack_patterns([])
    assert P.size == 0 and P_off.tolist() == [0]


# ---- the kernels' word comparison -----------------------------------------------------------------------------------
def _word(buf, end, p):
    """lcp_word: buf[p..p+3] as a little-endian word, bytes at or past `end` read as 0."""
    return sum(int(buf[p + k]) << (8 * k) for k in range(4) if p + k < end)


def word_compare(T, s, P, k0):
    """search_cmp_thread: suffix T[s:] against P (m >= 1) from byte min(k0, len) on; returns (sign, match)."""
    n, m = len(T), len(P)
    if s >= n:
        return -1, 0
    length = min(m, n - s)
    k = min(k0, length)
    while k < length:
        a, b = _word(T, n, s + k), _word(P, m, k)
        d = a ^ b
        if d:
            sh = ((d & -d).bit_length() - 1) & ~7  # __ffs(d) - 1, rounded down to its byte
            j = k + sh // 8
            if j >= length:
                break
            return (-1 if (a >> sh) & 0xFF < (b >> sh) & 0xFF else 1), j
        k += 4
    return (0 if length == m else -1), length


def byte_compare(T, s, P):
    n, m = len(T), len(P)
    if s >= n:
        return -1, 0
    j = 0
    while s + j < n and j < m and T[s + j] == P[j]:
        j += 1
    if j < m and s + j < n:
        return (-1 if T[s + j] < P[j] else 1), j
    return (0 if j == m else -1), j


def test_word_compare_random_words():
    rng = np.random.default_rng(3)
    for _ in range(3000):
        n = int(rng.integers(1, 24))
        sigma = int(rng.choice([2, 256]))
        T = rng.integers(0, sigma, n).astype(np.uint8)
        s = int(rng.integers(0, n + 2))
        m = int(rng.integers(1, 20))
        P = bytearray(rng.integers(0, sigma, m).astype(np.uint8).tobytes())
        if s < n and rng.random() < 0.7:  # mostly a prefix of the suffix, with one byte changed or cut
            P = bytearray(bytes(T[s:s + m]) + P[max(0, n - s):]) if rng.random() < 0.5 else bytearray(bytes(T[s:s + m]))
            if P and rng.random() < 0.5:
                P[int(rng.integers(0, len(P)))] ^= int(rng.integers(1, 256))
        if not P:
            continue
        want = byte_compare(T, s, P)
        assert word_compare(T, s, P, 0) == want, (T.tolist(), s, list(P))
        k0 = int(rng.integers(0, want[1] + 1))  # start anywhere within the bytes known to be equal
        assert word_compare(T, s, P, k0) == want


@pytest.mark.parametrize("zero", [False, True])
def test_word_compare_every_end_offset(zero):
    """Texts and patterns that end 0..8 bytes into the compared words, with equal bytes up to the end and 0x00 (the byte
    lcp_word pads with) as data: the lengths decide, never the padding."""
    fill = 0 if zero else 0x41
    for n in range(1, 17):
        T = np.full(n, fill, np.uint8)
        for s in range(n + 1):
            for m in range(1, 10):
                for extra in range(0, 9):
                    P = bytes([fill]) * m
                    assert word_compare(T, s, P, 0) == byte_compare(T, s, P)
                    if m > extra:
                        Q = bytearray(P)
                        Q[m - 1 - extra] ^= 1
                        assert word_compare(T, s, bytes(Q), 0) == byte_compare(T, s, bytes(Q))


# ---- arguments that need no device ----------------------------------------------------------------------------------
def test_null_context_is_earg():
    lib = bw.load_library()
    z8, z32, z64 = np.zeros(4, np.uint8), np.zeros(4, np.int32), np.zeros(2, np.uint64)
    assert lib.bwtc_cuda_sa_search(None, z8.ctypes.data, 4, z32.ctypes.data, 4, z8.ctypes.data, z64.ctypes.data, 1,
                                   z32.ctypes.data, z32.ctypes.data) == EARG
    assert lib.bwtc_cuda_sa_search_device(None, z8.ctypes.data, 4, z32.ctypes.data, 4, z8.ctypes.data, z64.ctypes.data,
                                          1, z32.ctypes.data, z32.ctypes.data) == EARG
    assert b"null context" in lib.bwtc_cuda_global_error()


def test_short_tier_cutoff_is_a_word_multiple():
    assert SEARCH_SHORT_BYTES % 4 == 0 and 4 <= SEARCH_SHORT_BYTES <= 128
