/* tests/lz77_oracle.c — test-only sequential restatement of bwtc_cuda_lz77 (include/bwtc_cuda.h, DESIGN.md §3.14).
 * Compiled by the tests into a temporary directory and loaded with ctypes.
 *
 * oracle_lz77: the greedy LZ77 parse of T from its suffix array SA (divsufsort's order): PSV / NSV of every row by a
 * stack, then, at each phrase start p only, the lengths l_P / l_N by direct comparison of T[p..] with T[SA[PSV]..] and
 * T[SA[NSV]..]; len = max(l_P, l_N), src = SA[PSV] if l_P >= l_N, else SA[NSV]; a literal (len 0) has src = T[p].
 * Writes at most capacity phrases and returns z (so capacity n is always enough), or -1 on bad arguments.
 * oracle_lz77_decode: rebuilds the text byte by byte (overlapping sources work); returns the bytes written, or -1 when a
 * source is not before its phrase or the output would pass n. */
#include <stdint.h>
#include <stdlib.h>

static uint32_t lcp_at(const uint8_t* T, uint32_t n, uint32_t a, uint32_t b) {
  uint32_t k = 0;
  while (a + k < n && b + k < n && T[a + k] == T[b + k]) ++k;
  return k;
}

int64_t oracle_lz77(const uint8_t* T, uint32_t n, const int32_t* SA, int32_t* src, int32_t* len, uint32_t capacity) {
  if (n == 0) return 0;
  if (!T || !SA) return -1;
  int64_t* psv = malloc((size_t)n * sizeof(int64_t));
  int64_t* nsv = malloc((size_t)n * sizeof(int64_t));
  int64_t* stk = malloc((size_t)n * sizeof(int64_t));
  uint32_t* isa = malloc((size_t)n * sizeof(uint32_t));
  if (!psv || !nsv || !stk || !isa) { free(psv); free(nsv); free(stk); free(isa); return -1; }
  int64_t top = 0;
  for (uint32_t r = 0; r < n; ++r) {  /* rows above r with a smaller SA value: the stack keeps them increasing */
    isa[SA[r]] = r;
    while (top > 0 && SA[stk[top - 1]] >= SA[r]) --top;
    psv[r] = top > 0 ? stk[top - 1] : -1;
    stk[top++] = r;
  }
  top = 0;
  for (uint32_t r = n; r-- > 0;) {
    while (top > 0 && SA[stk[top - 1]] >= SA[r]) --top;
    nsv[r] = top > 0 ? stk[top - 1] : -1;
    stk[top++] = r;
  }
  int64_t z = 0;
  for (uint32_t p = 0; p < n;) {
    const uint32_t r = isa[p];
    const uint32_t lp = psv[r] >= 0 ? lcp_at(T, n, p, (uint32_t)SA[psv[r]]) : 0;
    const uint32_t ln = nsv[r] >= 0 ? lcp_at(T, n, p, (uint32_t)SA[nsv[r]]) : 0;
    const uint32_t l = lp > ln ? lp : ln;
    if ((uint64_t)z < capacity) {
      len[z] = (int32_t)l;
      src[z] = l == 0 ? (int32_t)T[p] : lp >= ln ? SA[psv[r]] : SA[nsv[r]];
    }
    ++z;
    p += l ? l : 1;
  }
  free(psv); free(nsv); free(stk); free(isa);
  return z;
}

int64_t oracle_lz77_decode(const int32_t* src, const int32_t* len, int64_t z, uint8_t* out, uint32_t n) {
  uint64_t o = 0;
  for (int64_t k = 0; k < z; ++k) {
    if (len[k] <= 0) {
      if (o >= n || src[k] < 0 || src[k] > 255) return -1;
      out[o++] = (uint8_t)src[k];
      continue;
    }
    if (src[k] < 0 || (uint64_t)src[k] >= o || o + (uint64_t)len[k] > n) return -1;
    for (uint32_t j = 0; j < (uint32_t)len[k]; ++j, ++o) out[o] = out[(uint64_t)src[k] + j];
  }
  return (int64_t)o;
}
