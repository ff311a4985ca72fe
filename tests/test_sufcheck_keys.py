"""CPU restatement of the device-side sufcheck (DESIGN.md §3.11, bwt_kernels.cuh k_sa_perm / k_sa_order).

SA[0..n) is the suffix array of T (raw contract: implicit end sentinel, a suffix that is a prefix of another sorts
first) exactly when
  (1) it is a permutation of [0, n): every value in range, none held by two rows, and
  (2) for every r >= 1: (T[SA[r-1]], ISA'[SA[r-1]+1]) < (T[SA[r]], ISA'[SA[r]+1]), with ISA' the inverse of SA and
      ISA'[n] = -1 for the empty suffix.
Here both checks are restated in numpy, including which row the device reports (the smallest row failing (1) -- out of
range, or holding a value an earlier row holds -- else the smallest row failing (2)), and compared with brute-force
suffix sorting on every short text and on random mutants of true suffix arrays: the check accepts exactly the true SA."""
import itertools

import numpy as np

RANGE, DUP, ORDER = 1, 2, 3  # SA_BAD_RANGE / SA_BAD_DUP / SA_BAD_ORDER


def brute_sa(T):
    b = bytes(np.asarray(T, np.uint8))
    return np.array(sorted(range(len(b)), key=lambda i: b[i:]), dtype=np.int32)


def sufcheck(T, SA):
    """None if SA is the suffix array of T, else (row, reason) of the failure the device reports."""
    T = np.asarray(T, np.uint8)
    SA = np.asarray(SA, np.int64)
    n = T.size
    if n == 0:
        return None
    valid = (SA >= 0) & (SA < n)
    first = np.full(n, n, np.int64)  # ISA by atomicMin: the first row holding each value
    rows = np.arange(n)
    np.minimum.at(first, SA[valid], rows[valid])
    dup = np.zeros(n, bool)
    dup[valid] = first[SA[valid]] != rows[valid]
    bad1 = ~valid | dup
    if bad1.any():
        r = int(np.argmax(bad1))
        return (r, RANGE if not valid[r] else DUP)
    isa1 = np.zeros(n + 1, np.int64)  # ISA' + 1: 0 for the empty suffix
    isa1[SA] = rows + 1
    key = (T[SA].astype(np.int64) << 32) | isa1[SA + 1]
    bad2 = key[1:] <= key[:-1]
    if bad2.any():
        return (int(np.argmax(bad2)) + 1, ORDER)
    return None


def _texts(alphabet, max_len):
    for n in range(0, max_len + 1):
        for t in itertools.product(alphabet, repeat=n):
            yield np.array(t, np.uint8)


def test_accepts_every_true_suffix_array_of_short_texts():
    for alphabet, max_len in (((0, 1, 2), 7), ((0x00, 0xFF), 10), ((5,), 12)):
        for T in _texts(alphabet, max_len):
            assert sufcheck(T, brute_sa(T)) is None, T


def test_rejects_every_other_permutation_of_short_texts():
    """Exhaustive: for every text of length <= 5 over {0, 1, 2}, the only permutation the check accepts is the SA."""
    for T in _texts((0, 1, 2), 5):
        want = brute_sa(T)
        for p in itertools.permutations(range(T.size)):
            ok = sufcheck(T, np.array(p, np.int32)) is None
            assert ok == bool(np.array_equal(p, want)), (T, p)


def _mutants(SA, rng):
    n = SA.size
    out = []
    if n >= 2:
        for r in {0, n // 2, n - 2}:
            m = SA.copy()
            m[r], m[r + 1] = m[r + 1], m[r]
            out.append(("swap", m))
        m = np.roll(SA, 1)
        out.append(("rotate", m))
        m = SA.copy()
        m[rng.integers(n)] = SA[rng.integers(n)]
        out.append(("dup", m))
    for v in (n, -1, 2**31 - 1):
        m = SA.copy()
        m[rng.integers(n)] = v
        out.append(("range", m))
    return out


def test_random_mutants_of_true_suffix_arrays():
    rng = np.random.default_rng(1106)
    for trial in range(300):
        n = int(rng.integers(1, 200))
        sigma = int(rng.choice([1, 2, 4, 256]))
        T = rng.integers(0, sigma, n).astype(np.uint8)
        if trial % 3 == 0:  # long repeats
            T = np.tile(T[: max(1, n // 7)], 8)[:n]
        SA = brute_sa(T)
        assert sufcheck(T, SA) is None
        for kind, m in _mutants(SA, rng):
            want_ok = np.array_equal(m, SA)
            got = sufcheck(T, m)
            assert (got is None) == want_ok, (kind, T, m, got)
            if kind == "range":
                assert got[1] == RANGE
            if kind == "dup" and not want_ok:
                assert got[1] == DUP and m[got[0]] == m[np.flatnonzero(m == m[got[0]])[0]]


def test_reported_row_is_the_first_failure():
    T = np.frombuffer(b"mississippi", np.uint8)
    SA = brute_sa(T)
    m = SA.copy()
    m[0], m[1] = m[1], m[0]
    assert sufcheck(T, m) == (1, ORDER)
    m = SA.copy()
    m[7] = SA[2]
    assert sufcheck(T, m) == (7, DUP)
    m[9] = -1  # a range failure after a duplicate: the duplicate's row is smaller
    assert sufcheck(T, m) == (7, DUP)
    m[1] = 11
    assert sufcheck(T, m) == (1, RANGE)
