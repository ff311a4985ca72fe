/* tests/lcp_oracle.c -- TEST INFRASTRUCTURE, not product code: the checker the LCP tests compare the GPU engine with
 * (tests/test_lcp_keys.py compiles it into a temporary directory and loads it with ctypes).
 *
 * LCP array of T[0..N) given its suffix array, by Kasai, Lee, Arimura, Arikawa & Park (CPM 2001): LCP[0] = 0, LCP[r] = the
 * longest common prefix of suffixes SA[r-1] and SA[r], a comparison stopping at the end of T.  A plain sequential pass over
 * text positions with a rank array -- not the irreducible-row / max-scan method of the GPU engine.
 * Returns 0, or -2 on allocation failure. */
#include <stdint.h>
#include <stdlib.h>

int oracle_lcp(const uint8_t* T, uint32_t N, const int32_t* SA, int32_t* LCP) {
  if (N == 0) return 0;
  uint32_t* rank = (uint32_t*)malloc((size_t)N * sizeof(uint32_t));
  if (!rank) return -2;
  for (uint32_t r = 0; r < N; ++r) rank[SA[r]] = r;
  uint32_t h = 0;
  for (uint32_t i = 0; i < N; ++i) {
    const uint32_t r = rank[i];
    if (r == 0) { LCP[0] = 0; h = 0; continue; }
    const uint32_t j = (uint32_t)SA[r - 1];
    while (i + h < N && j + h < N && T[i + h] == T[j + h]) ++h;
    LCP[r] = (int32_t)h;
    if (h > 0) --h;
  }
  free(rank);
  return 0;
}
