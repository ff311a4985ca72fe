/* tests/sa_search_oracle.c -- TEST INFRASTRUCTURE, not product code: the checker the pattern-search tests compare the GPU
 * engine with (tests/test_sa_search_keys.py compiles it into a temporary directory and loads it with ctypes), and the CPU
 * baseline of tests/gpu_sa_search_probe.py.
 *
 * libdivsufsort's sa_search, one pattern after the other: a binary search that keeps the bytes the two ends of its
 * interval share with the pattern (the match-length heuristic) until it meets a row that starts with the pattern, then one
 * search on each side of that row for the ends of the run.  Not the two-bound search of the GPU engine.  Conventions of
 * bwtc_cuda_sa_search (include/bwtc_cuda.h): an SA entry outside [0, n) is the empty suffix, which sorts below every
 * non-empty pattern; a pattern is cut at n + 1 bytes; n == 0 or SAsize == 0 gives left = -1, size = 0; an empty pattern
 * gives left = 0, size = SAsize.  Offsets must not decrease.  Exact for an SA of suffixes in sorted order. */
#include <stdint.h>

/* Suffix s against P[0..m): < 0, 0, > 0 as the suffix sorts below, starts with, sorts above P.  *match: bytes known
 * equal on entry, bytes shared on return. */
static int compare(const uint8_t* T, uint32_t n, const uint8_t* P, uint32_t m, uint32_t s, uint32_t* match) {
  if (s >= n) {
    *match = 0;
    return -1;
  }
  uint32_t j = *match;
  if (j > n - s) j = n - s;
  int r = 0;
  while (s + j < n && j < m && (r = (int)T[s + j] - (int)P[j]) == 0) ++j;
  *match = j;
  return r == 0 ? -(j != m) : r;
}

static uint32_t min_u32(uint32_t a, uint32_t b) { return a < b ? a : b; }

/* One pattern; returns size, writes *idx. */
static uint32_t search_one(const uint8_t* T, uint32_t n, const int32_t* SA, uint32_t SAsize, const uint8_t* P, uint32_t m,
                           int32_t* idx) {
  uint32_t i = 0, j = 0, k = 0, lmatch = 0, rmatch = 0, size, half, match;
  int r;
  for (size = SAsize, half = size >> 1; size > 0; size = half, half >>= 1) {
    match = min_u32(lmatch, rmatch);
    r = compare(T, n, P, m, (uint32_t)SA[i + half], &match);
    if (r < 0) {
      i += half + 1;
      half -= (size & 1) ^ 1;
      lmatch = match;
    } else if (r > 0) {
      rmatch = match;
    } else {
      uint32_t lsize = half, rsize = size - half - 1, llmatch, lrmatch, rlmatch, rrmatch;
      j = i;
      k = i + half + 1;
      for (llmatch = lmatch, lrmatch = match, half = lsize >> 1; lsize > 0; lsize = half, half >>= 1) {
        lmatch = min_u32(llmatch, lrmatch);
        r = compare(T, n, P, m, (uint32_t)SA[j + half], &lmatch);
        if (r < 0) {
          j += half + 1;
          half -= (lsize & 1) ^ 1;
          llmatch = lmatch;
        } else {
          lrmatch = lmatch;
        }
      }
      for (rlmatch = match, rrmatch = rmatch, half = rsize >> 1; rsize > 0; rsize = half, half >>= 1) {
        rmatch = min_u32(rlmatch, rrmatch);
        r = compare(T, n, P, m, (uint32_t)SA[k + half], &rmatch);
        if (r <= 0) {
          k += half + 1;
          half -= (rsize & 1) ^ 1;
          rlmatch = rmatch;
        } else {
          rrmatch = rmatch;
        }
      }
      break;
    }
  }
  *idx = (int32_t)(k > j ? j : i);
  return k - j;
}

/* Patterns first .. first + count - 1 of the batch (P_off: offsets into P); results at left[0..count), size[0..count). */
void oracle_sa_search(const uint8_t* T, uint32_t n, const int32_t* SA, uint32_t SAsize, const uint8_t* P,
                      const uint64_t* P_off, uint32_t first, uint32_t count, int32_t* left, int32_t* size) {
  for (uint32_t q = 0; q < count; ++q) {
    const uint64_t beg = P_off[first + q], end = P_off[first + q + 1];
    const uint64_t full = end - beg;
    const uint32_t m = full > (uint64_t)n + 1 ? n + 1 : (uint32_t)full;
    if (n == 0 || SAsize == 0) {
      left[q] = -1;
      size[q] = 0;
    } else if (m == 0) {
      left[q] = 0;
      size[q] = (int32_t)SAsize;
    } else {
      size[q] = (int32_t)search_one(T, n, SA, SAsize, P + beg, m, &left[q]);
    }
  }
}
