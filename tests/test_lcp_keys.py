"""CPU restatement of the device-side LCP construction (DESIGN.md §3.12, bwt_kernels.cuh k_lcp_*).

Given the suffix array SA of T (raw contract: implicit end sentinel), with i = SA[r] and j = SA[r-1]:
  (1) row r >= 1 is irreducible when i == 0 or j == 0 or T[i-1] != T[j-1]; only those rows compare T[i..] with T[j..]
      and store X[i] = i + lcp; row 0 stores X[SA[0]] = SA[0]; every other X[i] is 0;
  (2) a comparison runs up to LCP_SHORT_BYTES bytes in one thread, then in windows [K 2^w, K 2^(w+1)) (the long tier);
  (3) PLCP[i] = maxscan(X)[i] - i;
  (4) LCP[r] = PLCP[SA[r]].
Here the four steps are restated in numpy and compared with brute-force LCPs on every short text and on random texts,
the comparison work is checked against the Kärkkäinen-Manzini-Puglisi bound, and oracle_lcp (the sequential Kasai of
tests/lcp_oracle.c that the GPU tests compare with) is pinned to brute force on the same texts."""
import atexit
import ctypes
import itertools
import math
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_sufcheck_keys import brute_sa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _constant(name):
    src = open(os.path.join(ROOT, "bwtc_b200", "csrc", "bwt_kernels.cuh")).read()
    return int(re.search(rf"constexpr uint32_t {name} = (\d+);", src).group(1))


LCP_SHORT_BYTES = _constant("LCP_SHORT_BYTES")
LCP_SEG_BYTES = _constant("LCP_SEG_BYTES")


_ORACLE = []


def _oracle_lib():
    """tests/lcp_oracle.c, compiled once per process into a temporary directory (the tree may be read-only)."""
    if not _ORACLE:
        cc = shutil.which("gcc") or shutil.which("cc")
        assert cc, "no C compiler for tests/lcp_oracle.c"
        tmp = tempfile.mkdtemp(prefix="lcp_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "liblcp_oracle.so")
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-std=c99", "-Wall", "-o", out,
                        os.path.join(ROOT, "tests", "lcp_oracle.c")], check=True)
        lib = ctypes.CDLL(out)
        lib.oracle_lcp.restype = ctypes.c_int
        lib.oracle_lcp.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p]
        _ORACLE.append(lib)
    return _ORACLE[0]


def oracle_lcp(T, SA):
    """The sequential Kasai LCP of T given its suffix array SA (int32[T.size])."""
    T = np.ascontiguousarray(T, np.uint8)
    SA = np.ascontiguousarray(SA, np.int32)
    LCP = np.empty(T.size, np.int32)
    assert _oracle_lib().oracle_lcp(T.ctypes.data, T.size, SA.ctypes.data, LCP.ctypes.data) == 0
    return LCP


def brute_lcp(T, SA):
    b = bytes(np.asarray(T, np.uint8))
    out = np.zeros(len(b), np.int32)
    for r in range(1, len(b)):
        x, y = b[SA[r - 1]:], b[SA[r]:]
        k = 0
        while k < min(len(x), len(y)) and x[k] == y[k]:
            k += 1
        out[r] = k
    return out


def lcp_model(T, SA, K=LCP_SHORT_BYTES):
    """Steps (1)-(4).  Returns LCP and the work: irreducible rows, bytes compared (each comparison up to and including its
    first mismatch, or to the end of the text), pairs that left the short tier, and the windows each of those reached."""
    T = np.asarray(T, np.uint8)
    SA = np.asarray(SA, np.int64)
    n = T.size
    X = np.zeros(n, np.int64)
    work = {"irreducible": 0, "bytes": 0, "long": 0, "windows": 0}
    if n == 0:
        return np.zeros(0, np.int32), work
    X[SA[0]] = SA[0]
    for r in range(1, n):
        i, j = int(SA[r]), int(SA[r - 1])
        if i != 0 and j != 0 and T[i - 1] == T[j - 1]:
            continue
        work["irreducible"] += 1
        limit = n - max(i, j)
        d = np.flatnonzero(T[i:i + limit] != T[j:j + limit])
        lcp = int(d[0]) if d.size else limit
        work["bytes"] += min(lcp + 1, limit)
        if lcp >= K and limit > K:
            work["long"] += 1
            w = 0  # window w covers [K 2^w, K 2^(w+1)); the pair goes on while a window holds no mismatch
            while True:
                work["windows"] += 1
                hi = K << (w + 1)
                if lcp < hi or hi >= limit:
                    break
                w += 1
        X[i] = i + lcp
    PLCP = np.maximum.accumulate(X) - np.arange(n)
    return PLCP[SA].astype(np.int32), work


def _texts(alphabet, max_len):
    for n in range(1, max_len + 1):
        for t in itertools.product(alphabet, repeat=n):
            yield np.array(t, np.uint8)


def _random_texts():
    rng = np.random.default_rng(2009)
    for trial in range(300):
        sigma = int(rng.integers(1, 5))
        n = int(rng.integers(1, 400))
        T = rng.integers(0, sigma, n).astype(np.uint8)
        if trial % 5 == 0:  # long repeats: copies of one random string
            s = rng.integers(0, sigma, int(rng.integers(1, 80))).astype(np.uint8)
            T = np.tile(s, n // s.size + 1)[:n].copy()
        yield T


@pytest.mark.parametrize("alphabet", [(0, 1, 2), (0x00, 0xFF)])
def test_every_short_text(alphabet):
    for T in _texts(alphabet, 8):
        SA = brute_sa(T)
        got, _ = lcp_model(T, SA)
        assert np.array_equal(got, brute_lcp(T, SA)), T.tolist()


def test_random_texts():
    for T in _random_texts():
        SA = brute_sa(T)
        got, _ = lcp_model(T, SA)
        assert np.array_equal(got, brute_lcp(T, SA)), T.tolist()


def test_small_tier_threshold_reaches_the_windows():
    """With a small K the windows run on short texts too: the result does not depend on where the tiers split."""
    for T in itertools.chain(_random_texts(), [np.full(300, 7, np.uint8)]):
        SA = brute_sa(T)
        want = brute_lcp(T, SA)
        for K in (1, 2, 4):
            got, _ = lcp_model(T, SA, K)
            assert np.array_equal(got, want), (K, T.tolist())


def test_comparison_work_bound():
    """Bytes compared stay within 2 n log2 n + n (the irreducible LCPs sum to at most 2 n log2 n, plus one mismatching
    byte per row); a single repeated byte compares once, n - 1 bytes, and that pair runs through every window."""
    texts = list(_random_texts()) + [T for T in _texts((0, 1), 10)]
    for T in texts:
        n = T.size
        _, work = lcp_model(T, brute_sa(T))
        assert work["bytes"] <= 2 * n * math.log2(max(n, 2)) + n, (T.tolist(), work)
    n = 1000
    T = np.full(n, 0x61, np.uint8)
    SA = np.arange(n - 1, -1, -1)
    lcp, work = lcp_model(T, SA)
    assert np.array_equal(lcp, np.arange(n))
    assert work["irreducible"] == 1 and work["bytes"] == n - 1 and work["long"] == 1
    assert work["windows"] == math.ceil(math.log2((n - 1) / LCP_SHORT_BYTES))


def test_oracle_lcp_equals_brute_force():
    texts = itertools.chain(_texts((0, 1, 2), 7), _texts((0x00, 0xFF), 8), _random_texts())
    for T in texts:
        SA = brute_sa(T)
        assert np.array_equal(oracle_lcp(T, SA), brute_lcp(T, SA)), T.tolist()
