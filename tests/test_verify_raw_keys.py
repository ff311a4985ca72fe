"""CPU restatement of the generalised inversion that verifies a raw forward transform (DESIGN.md §3.10, ibwt_kernels.cuh).

A raw text T of N bytes ends in an arbitrary byte c = T[N-1]; its output U has U[pidx] unwritten.  The keys
key(pidx) = c, key(r) = L[r] + [L[r] >= c] sort every row to its F-row, the end-of-text row to C[c] (the row of suffix
N - 1).  The walk counts its splitters from that anchor, recovers F as v - [v > c] and checks, at every sampled text
position q = N - j x, that the row is LFpowers[j].  With c = 0 the keys and the anchor are the block contract's own.
Here the kernels' steps (keys, stable sort, C table, walk 1, pointer jumping, walk 2, comparison) are restated in numpy
and run on oracle outputs."""
import numpy as np

import bwtc_b200 as bw
from test_gpu_raw_contract import KINDS, LAST_BYTE_FORMS, last_byte_form

K = 32  # INV_K


def inv_keys(L, eob, c):
    key = L.astype(np.int64) + (L >= c)
    key[eob] = c
    return key


def block_keys_today(out, eob):
    """k_inv_keys as the block contract has always keyed it: L + 1, 0 at eob, row N - 1 from out[eob]."""
    n = out.size
    L = np.append(out, out[eob] if eob < n else 0).astype(np.int64)
    key = L + 1
    key[eob] = 0
    return key, L


def verify(U, T_body, LF, c, nLF=None):
    """The device check, restated: True when U with end-of-text row LF[0] and last byte c restores T_body (N - 1 bytes)
    and every LF[j] (1 <= j < nLF) is the row the walk visits at text position N - j floor(N / nLF).  Returns
    (ok, restored, rows at the sampled positions)."""
    N = U.size
    eob = int(LF[0])
    nLF = LF.size if nLF is None else nLF
    key = inv_keys(U, eob, c)
    psi = np.argsort(key, kind="stable")  # psi[g] = the L-row of F-row g
    C = np.searchsorted(np.sort(key), np.arange(258), side="left")  # C[v] = keys below v
    a = int(C[c])
    S = -(-N // K)
    # walk 1: splitter j at row (a + j K) mod N follows psi to the next splitter
    nxt = np.empty(S, np.int64)
    ln = np.empty(S, np.int64)
    for j in range(S):
        g, t = (a + j * K) % N, 0
        while True:
            g = int(psi[g])
            t += 1
            x = (g - a) % N
            if x % K == 0 or t >= N:
                break
        to = x // K
        nxt[j] = -1 if to == 0 else to
        ln[j] = t
    # pointer jumping, ceil(log2 S) rounds
    dist, nx = ln.copy(), nxt.copy()
    span = 1
    while span < S:
        live = nx >= 0
        d2 = dist.copy()
        d2[live] += dist[nx[live]]
        n2 = np.full(S, -1, np.int64)
        n2[live] = nx[nx[live]]
        dist, nx = d2, n2
        span <<= 1
    cycle_ok = ln.sum() == N and (nx < 0).all()
    # walk 2
    out = np.zeros(N - 1, np.int64)
    x = N // nLF
    sampled = {N - j * x: j for j in range(1, nLF)}
    rows = {}
    for j in range(S):
        g = (a + j * K) % N
        q = (2 * N - 1 - int(dist[j])) % N
        for _ in range(int(ln[j])):
            if q in sampled:
                rows[sampled[q]] = g
            if q < N - 1:
                v = int(np.searchsorted(C, g, side="right")) - 1  # the largest v with C[v] <= g
                out[N - 2 - q] = v - (v > c)
            g = int(psi[g])
            q = (q + 1) % N
    restored = out[::-1].astype(np.uint8)
    lf_ok = all(rows.get(j) == int(LF[j]) for j in range(1, nLF))
    return bool(cycle_ok and lf_ok and np.array_equal(restored, T_body)), restored, rows


def _raw_cases():
    rng = np.random.default_rng(501)
    for kind in KINDS:
        for form in LAST_BYTE_FORMS:
            R = np.ascontiguousarray(bw.generate(kind, 4999, seed=7)[::-1])
            yield f"{kind}/{form}", last_byte_form(R, form, rng), 8
    for n in range(2, 301):
        sigma = int(rng.choice([1, 2, 4, 256]))
        T = rng.integers(0, sigma, n).astype(np.uint8) + (0 if sigma == 256 else int(rng.integers(0, 200)))
        if n % 3 == 0:
            T[-1] = rng.integers(0, 256)
        yield f"n={n}", T, [1, 8, 256][n % 3]
    for n in (2, 3, 31, 32, 33, 257, 1000):
        for v in (0, 7, 255):
            yield f"equal n={n} v={v}", np.full(n, v, np.uint8), 8
    for nLF in (1, 8, 256):
        T = np.append(rng.integers(0, 4, 2999), 1).astype(np.uint8)
        yield f"nLF={nLF}", T, nLF


def test_generalised_keys_restore_raw_texts_and_sample_lfpowers(oracle):
    seen_c = set()
    for what, T, nLF in _raw_cases():
        nLF = min(nLF, T.size)
        rc, U, LF, _ = oracle.raw(T, nLF)
        c = int(T[-1])
        seen_c.add(c)
        ok, restored, rows = verify(U, T[:-1], LF, c)
        assert np.array_equal(restored, T[:-1]), what
        assert all(rows[j] == LF[j] for j in range(1, nLF)), what
        assert ok, what
    assert len(seen_c) > 50


def test_zero_keys_are_todays_block_keys(oracle):
    """c = 0 on the block contract: the generalised keys equal the keying the inverse has always used, the anchor is row 0
    (the splitters of the plain inverse), and the check accepts the output with all its LFpowers."""
    for kind in KINDS:
        for n in (1, 2, 33, 300, 5000):
            x = bw.generate(kind, n, seed=600 + n)
            out, LF, _ = oracle.block(x, 8)
            eob = int(LF[0])
            today, L = block_keys_today(out, eob)
            key = inv_keys(L, eob, 0)
            assert np.array_equal(key, today), (kind, n)
            assert np.searchsorted(np.sort(key), 0) == 0
            ok, restored, _ = verify(L.astype(np.uint8), x[::-1].copy(), LF, 0)
            assert ok and np.array_equal(restored[::-1], x), (kind, n)


def test_mutated_raw_outputs_fail_the_check(oracle):
    """A changed byte at a row other than pidx, a swap of unequal bytes, a moved pidx and a wrong LFpowers[j] each fail;
    the unchanged output passes."""
    rng = np.random.default_rng(503)
    fails = {"byte": 0, "swap": 0, "pidx": 0, "lf": 0}
    for what, T, nLF in _raw_cases():
        N = T.size
        if N < 40 or np.unique(T[:-1]).size < 2:
            continue
        nLF = min(nLF, N)
        _, U, LF, _ = oracle.raw(T, nLF)
        c, p = int(T[-1]), int(LF[0])
        assert verify(U, T[:-1], LF, c)[0], what
        rows = [r for r in range(N) if r != p]
        m = U.copy()
        r = int(rng.choice(rows))
        m[r] ^= 1
        assert not verify(m, T[:-1], LF, c)[0], (what, "byte")
        fails["byte"] += 1
        i = int(rng.choice(rows))
        js = [j for j in rows if U[j] != U[i]]
        if js:
            m = U.copy()
            j = int(rng.choice(js))
            m[i], m[j] = m[j], m[i]
            assert not verify(m, T[:-1], LF, c)[0], (what, "swap")
            fails["swap"] += 1
        lf = LF.copy()
        lf[0] = (p + 1 + int(rng.integers(N - 1))) % N
        assert not verify(U, T[:-1], lf, c)[0], (what, "pidx")
        fails["pidx"] += 1
        if nLF > 1:
            lf = LF.copy()
            j = int(rng.integers(1, nLF))
            lf[j] ^= 1
            assert not verify(U, T[:-1], lf, c)[0], (what, "lf")
            fails["lf"] += 1
    assert all(v >= 10 for v in fails.values()), fails
