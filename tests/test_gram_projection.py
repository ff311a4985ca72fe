"""CPU check of the arithmetic behind the gram mode of round 0 (DESIGN.md §3.2, bwt_kernels.cuh GramParams): for 6-bit and
3-bit codes every digit histogram of the round-0 radix sort is a projection of ONE histogram of the keys' low 12 bits,
plus u head terms and minus u tail terms.  The (u, s) choice below is the one plan_histograms makes (bwt_engine.cu, "Gram mode");
the kernels themselves are checked bit-exactly on the GPU (tests/test_gpu_parity.py)."""
import numpy as np
import pytest

GRAM_BITS = 12


def _keys(codes, c, b, r=0):
    """key(i) = c codes starting at i, most significant first, then the top r bits of the next code; zero padding past the
    end (k_pack_round0).  Returns (key, E) with E = the c exact characters."""
    n = codes.size
    padded = np.concatenate([codes.astype(np.uint64), np.zeros(c + 1, np.uint64)])
    E = np.zeros(n, np.uint64)
    for j in range(c):
        E = (E << np.uint64(b)) | padded[j:j + n]
    key = E
    if r:
        key = (E << np.uint64(r)) | (padded[c:c + n] >> np.uint64(b - r))
    return key, E


def _plan(c, b, rb, r=0):
    """(u, s) per digit, in the coordinates of E: digit p of the key = E bits [rb p - r, rb p - r + rb).  u = -1: the lowest
    digit reaches into the partial character — its window is the low window of E(i + 1)."""
    keybits = c * b + r
    npass = -(-keybits // rb)
    W = GRAM_BITS // b
    plan = []
    for p in range(npass):
        lo = rb * p - r
        if lo < 0:
            u, s = -1, lo + b
        else:
            u = min(lo // b, c - W)
            s = lo - b * u
        assert s + rb <= GRAM_BITS or rb * p + rb > keybits, "digit outside its 12-bit window"
        plan.append((u, s))
    return plan


@pytest.mark.parametrize("b,c,r", [(6, 2, 0), (6, 3, 0), (6, 5, 0), (6, 9, 0), (6, 10, 0), (3, 4, 0), (3, 5, 0), (3, 10, 0),
                                   (3, 12, 0), (3, 21, 0), (6, 10, 4), (6, 5, 2), (6, 2, 4), (6, 9, 2), (6, 6, 4), (3, 21, 1),
                                   (3, 5, 1), (3, 10, 2), (6, 7, 5), (6, 3, 1)])
@pytest.mark.parametrize("rb", [8, 9])
def test_digit_histograms_are_projections_of_the_gram_histogram(b, c, r, rb):
    if (c * b + r) % rb and r:  # the engine only adds partial bits that fill the last digit
        r_fill = (-(c * b)) % rb
        if r_fill >= b or r_fill == 0:
            pytest.skip("no partial bits for this shape")
        r = r_fill
    rng = np.random.default_rng(100 * b + c + rb + 7 * r)
    dmask = (1 << rb) - 1
    for n, tail in ((65, 0), (1000, (1 << b) - 1), (4099, 1)):
        codes = rng.integers(0, 1 << b, n).astype(np.uint64)
        codes[-30:] = tail
        key, E = _keys(codes, c, b, r)
        low = (E & np.uint64((1 << GRAM_BITS) - 1)).astype(np.int64)  # the engine counts (key >> r) & 0xFFF
        G = np.bincount(low, minlength=1 << GRAM_BITS)
        g = np.arange(1 << GRAM_BITS)
        for p, (u, s) in enumerate(_plan(c, b, rb, r)):
            direct = np.bincount(((key >> np.uint64(rb * p)) & np.uint64(dmask)).astype(np.int64), minlength=dmask + 1)
            proj = np.bincount((g >> s) & dmask, weights=G, minlength=dmask + 1).astype(np.int64)
            if u >= 0:
                for i in range(u):  # head: suffixes 0..u-1 are not covered by a slid window; tail: the last u have no partner
                    proj[int((int(key[i]) >> (rb * p)) & dmask)] += 1
                    proj[(int(low[n - 1 - i]) >> s) & dmask] -= 1
            else:  # window of E(i + 1): suffix 0's own window is not anybody's, the all-padding window of "suffix n" is
                proj[(int(low[0]) >> s) & dmask] -= 1
                proj[0] += 1
            assert (proj == direct).all(), (n, p, u, s)
