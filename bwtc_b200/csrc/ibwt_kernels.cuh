// bwtc_b200/csrc/ibwt_kernels.cuh — hand-written sm_100a kernels of the INVERSE Burrows-Wheeler transform
// (SURVEY.md §8f row f4).  Replaces InverseBWTransform::doTransform / MtlSaInverseBWTransform
// (bwtransforms/InverseBWT.hpp:45-55, InverseBWT.cpp:47-51, MtlSaInverseBWT.cpp:246-362) — not a port of MTL-SA.
//
// Convention (same as the forward path, DESIGN.md §1): T' = reverse(X) . $, N = n + 1, L[r] = T'[SA[r] - 1],
// eob = LFpowers[0] = rank of suffix 0 (L[eob] is the sentinel).  The reference inverts by following LF from row 0
// (FastInverseBWTransform, InverseBWT.cpp:58-115) — one dependent random access per byte, inherently serial; its MTL-SA
// variant runs a handful of such chains (the LFpowers starting points) on CPU threads.  A GPU needs ~10^5 independent
// chains, so the starting points are made on the device instead:
//   1. k_inv_keys     key[r] = L[r] + 1 (0 for the sentinel row; a raw text's last byte c in general, see below),
//                     9 significant bits (+ the block number of a batch above them), + both digit histograms
//   2. k_radix_pass   x 2 (the forward path's one-sweep LSD pass, stable): Psi[g] = the L-row of F-row g, i.e. the
//                     rank of the suffix that starts one position LATER in T' — walking Psi walks T' forwards
//   3. k_inv_ctable   C[c] = number of key values < c (F[g] is recovered by a search in C, no F array in memory)
//   4. k_inv_walk1    every K-th rank (K = 32) is a SPLITTER; each splitter follows Psi to the next splitter: (next, length)
//   5. k_inv_jump     x ceil(log2 S): pointer jumping over the S = N/K splitters -> distance of each to the end of the
//                     cycle opened at rank 0 (suffix N-1), i.e. its text position
//   6. k_inv_walk2    each splitter walks its stretch again and writes X[n-1-q] = F[rank(q)] for its text positions q;
//                     it also decides whether L is the BWT of any text at all (Psi one cycle, DESIGN.md §3.7)
// Two passes of N dependent-per-chain but mutually independent random reads with ~N/K chains in flight: bound by the
// L2/DRAM random-access rate, not by latency.  LFpowers[1..] are not needed (the device makes far denser samples); the
// verification of a forward transform (walk kernels with VERIFY) checks them against the rows the walk visits.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bwtc_b200 {

#ifndef BWTC_INV_K
#define BWTC_INV_K 32
#endif
constexpr uint32_t INV_K = BWTC_INV_K;   // splitter spacing in rank space = average chain length.  Measured (32 MiB Markov, one
                                         // block): 128 -> 2.63 ms, 64 -> 2.29 ms, 32 -> 2.00 ms: shorter chains even out the
                                         // geometric spread of chain lengths that leaves lanes idle (profiles/r02_summary.md)
constexpr uint32_t INV_NIL = 0xFFFFFFFFu;
// ctrl[2..3]: bit k set = block k of the inversion is corrupt (its Psi is not one cycle: not the BWT of any text with that
// end-of-block row) or, when a forward transform is verified, does not restore its text.  Zeroed with the sticky words.
constexpr int CTR_INV_BAD = 2;
__device__ __forceinline__ void inv_mark_bad(uint32_t* ctrl, uint32_t k) { atomicOr(&ctrl[CTR_INV_BAD + (k >> 5)], 1u << (k & 31u)); }

// Batch of blocks inverted as ONE problem (DESIGN.md §3.7), the layout of the forward batch (§3.6): B blocks of n0 bytes,
// the last one n_last <= n0 bytes; block k has N_k = n_k + 1 rows and owns rows [k R, k R + N_k) with R = n0 + 1, its
// bytes sit at in + k n0 (and its result at out + k n0).  Keys are (k << 9) | (L + 1): the block number on top makes the
// stable 2-digit sort keep every block's F-rows inside its own row range, so Psi maps each block into itself, and each
// block's sentinel row has a key of its own (k << 9) — no byte value is reserved, unlike the forward batch.
// A single block is B = 1, R = N_last = N (k = 0 everywhere: the kernels do exactly what they did before batching).
constexpr uint32_t INV_MAX_BLOCKS = 64;  // = BWTC_CUDA_MAX_BATCH
struct InvShape {
  uint32_t nblocks;  // B
  uint32_t R;        // row stride (B = 1: N)
  uint32_t n0;       // byte stride of the output blocks (B = 1: unused)
  uint32_t istride;  // byte stride of the input blocks: n0, or R for the output of a forward batch (B = 1: unused)
  uint32_t N_last;   // rows of the last block
  uint32_t S0;       // splitters of a full block (ceil(R / INV_K)) ...
  uint32_t S_last;   // ... and of the last block
  uint32_t eob[INV_MAX_BLOCKS];  // per block: the end-of-block row (LFpowers[0]) ...
  const uint32_t* d_eob;         // ... or, if not null, read on the device from d_eob[256 k] (a forward transform's LFpowers rows)
  uint8_t eot[INV_MAX_BLOCKS] = {};  // per block: the byte c of its end-of-text row (0 except when a raw forward is verified)
  uint32_t nLF = 1, nLF_last = 1;    // verification only: LFpowers per full block / in the last block, in the d_eob rows
};
__device__ __forceinline__ uint32_t inv_eob(const InvShape& sh, uint32_t k) { return sh.d_eob ? sh.d_eob[256u * k] : sh.eob[k]; }
__host__ __device__ __forceinline__ uint32_t inv_rows(const InvShape& sh) { return (sh.nblocks - 1u) * sh.R + sh.N_last; }
__host__ __device__ __forceinline__ uint32_t inv_splitters(const InvShape& sh) { return (sh.nblocks - 1u) * sh.S0 + sh.S_last; }

// key[r] = L[r] + [L[r] >= c], c at the end-of-text row eob, block number k (= blockIdx.y) above bit 9; c = sh.eot[k] is
// the text's last byte, 0 for a sentinel-terminated text (key = L + 1, 0 at eob).  The value c belongs to the eob row alone,
// rows with L < c keep their bucket, rows with L >= c move up by the one F entry of the last suffix: the stable sort puts
// every row at its F-row, the eob row at C[c], the row of suffix N_k - 1 (DESIGN.md §3.10).  Row N_k-1 holds, in the block
// contract, the byte the forward transform moved into the hole (out[eob] = L[N-1], BWTransform.cpp:60); in the raw
// contract (single block only) in[N-1] itself.
// hist[0..255] = histogram of key & 0xFF (all blocks), hist[256 + 2k + 1] = keys of block k with value 256 (byte 0xFF);
// k_inv_ctable derives hist[256 + 2k] from it.  bhist (batch only, else nullptr): [k][256] the low-byte histogram per block.
__global__ void __launch_bounds__(256) k_inv_keys(const uint8_t* __restrict__ in, const InvShape sh, int block_mode,
                                                  uint32_t* __restrict__ keys, uint32_t* __restrict__ hist,
                                                  uint32_t* __restrict__ bhist) {
  __shared__ uint32_t s_lo[256];
  __shared__ uint32_t s_hi;
  s_lo[threadIdx.x] = 0;
  if (threadIdx.x == 0) s_hi = 0;
  __syncthreads();
  const uint32_t k = blockIdx.y;
  const uint32_t N = (k + 1u == sh.nblocks) ? sh.N_last : sh.R, eob = inv_eob(sh, k);
  const uint8_t* __restrict__ ink = in + (size_t)k * sh.istride;
  uint32_t* __restrict__ kk = keys + (size_t)k * sh.R;
  const uint32_t top = k << 9, c = sh.eot[k];
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < N; r += gridDim.x * blockDim.x) {
    uint32_t key;
    if (r == eob) {
      key = c;
    } else {
      key = (r == N - 1u && block_mode) ? (uint32_t)ink[eob] : (uint32_t)ink[r];
      key += key >= c ? 1u : 0u;
    }
    kk[r] = top | key;
    atomicAdd(&s_lo[key & 0xFFu], 1u);
    if (key >> 8) atomicAdd(&s_hi, 1u);
  }
  __syncthreads();
  const uint32_t v = s_lo[threadIdx.x];
  if (v) {
    atomicAdd(&hist[threadIdx.x], v);
    if (bhist) atomicAdd(&bhist[k * 256u + threadIdx.x], v);
  }
  if (threadIdx.x == 0) {
    if (s_hi) atomicAdd(&hist[256 + 2u * k + 1u], s_hi);
  }
}

// One CTA per block k.  hist[256 + 2k] = N_k - hist[256 + 2k + 1] (the second digit pass needs the full histogram of its
// digit, key >> 8 = 2k + (value >> 8)); C[k][0..257]: C[k][v] = k R + number of keys of block k below value v, i.e. the
// F-row where value v starts in block k (key values are 0..256).
__global__ void k_inv_ctable(uint32_t* __restrict__ hist, const uint32_t* __restrict__ bhist, const InvShape sh,
                             uint32_t* __restrict__ C) {
  if (threadIdx.x != 0) return;
  const uint32_t k = blockIdx.x;
  const uint32_t N = (k + 1u == sh.nblocks) ? sh.N_last : sh.R;
  const uint32_t* lo = bhist ? bhist + (size_t)k * 256 : hist;
  uint32_t* Ck = C + (size_t)k * 258;
  const uint32_t n256 = hist[256 + 2u * k + 1u];  // keys with value 256 (byte 0xFF)
  hist[256 + 2u * k] = N - n256;
  uint32_t acc = k * sh.R;
  for (uint32_t v = 0; v <= 256; ++v) {
    Ck[v] = acc;
    uint32_t cnt;
    if (v == 0) cnt = lo[0] - n256;      // low digit 0 is shared by key 0 (the sentinel) and key 256
    else if (v == 256) cnt = n256;
    else cnt = lo[v];
    acc += cnt;
  }
  Ck[257] = acc;
}

// Psi[g] = iota_top - vals[g] (the radix pass numbered the rows downwards, see k_radix_pass IOTA).
__device__ __forceinline__ uint32_t inv_psi(const uint32_t* __restrict__ vals, uint32_t iota_top, uint32_t g) {
  return iota_top - vals[g];
}

// Splitter rows are counted from the block's anchor a, the F-row of suffix N_k - 1: local row (a + j K) mod N_k is splitter
// j.  The plain inverse has a = 0 (c = 0: the eob row sorts first); a verified forward (VERIFY) reads a = C[k][c] - k R.
template <bool VERIFY>
__device__ __forceinline__ uint32_t inv_anchor(const uint32_t* C, const InvShape& sh, uint32_t k) {
  return VERIFY ? C[(size_t)k * 258 + sh.eot[k]] - k * sh.R : 0u;
}
// local row x -> its distance from the anchor (mod N)
template <bool VERIFY>
__device__ __forceinline__ uint32_t inv_from_anchor(uint32_t x, uint32_t a, uint32_t N) {
  return VERIFY ? (x >= a ? x - a : x + N - a) : x;
}

// Grid (ceil(S0 / 256), B).  Splitter j of block k = local row (a + j K) mod N_k, global index k S0 + j.  Follow Psi until
// the next splitter of the block: nxt = its index, len = steps taken (>= 1).  The splitter whose successor is the block's
// splitter 0 gets nxt = INV_NIL: each block's cycle is opened at its anchor (= suffix N_k - 1).
template <bool VERIFY>
__global__ void __launch_bounds__(256) k_inv_walk1(const uint32_t* __restrict__ vals, const InvShape sh,
                                                   const uint32_t* __restrict__ C, uint32_t* __restrict__ nxt,
                                                   uint32_t* __restrict__ len, const uint32_t* __restrict__ ctrl) {
  const uint32_t k = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
  const bool last = k + 1u == sh.nblocks;
  if (j >= (last ? sh.S_last : sh.S0) || ctrl[0]) return;  // ctrl[CTR_ERR]: a digit pass failed, Psi is not trustworthy
  const uint32_t N = last ? sh.N_last : sh.R, base = k * sh.R, top = inv_rows(sh) - 1u;
  const uint32_t a = inv_anchor<VERIFY>(C, sh, k);
  uint32_t g = base + (VERIFY ? (a + j * INV_K) % N : j * INV_K), t = 0, x;
  do {
    g = inv_psi(vals, top, g);
    ++t;
    x = inv_from_anchor<VERIFY>(g - base, a, N);
  } while (x % INV_K != 0u && t < N);
  const uint32_t to = x / INV_K;
  const uint32_t s = k * sh.S0 + j;
  nxt[s] = (to == 0u) ? INV_NIL : k * sh.S0 + to;
  len[s] = t;
}

// One pointer-jumping round: dist_out[s] = dist_in[s] + dist_in[nxt_in[s]], nxt_out[s] = nxt_in[nxt_in[s]].
__global__ void __launch_bounds__(256) k_inv_jump(const uint32_t* __restrict__ nxt_in, const uint32_t* __restrict__ dist_in,
                                                  uint32_t S, uint32_t* __restrict__ nxt_out, uint32_t* __restrict__ dist_out,
                                                  const uint32_t* __restrict__ ctrl) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S || ctrl[CTR_ERR]) return;  // sticky error: walk1 did not run, nxt_in holds stale indices
  const uint32_t nx = nxt_in[s];
  uint32_t d = dist_in[s], n2 = INV_NIL;
  if (nx != INV_NIL) {
    d += dist_in[nx];
    n2 = nxt_in[nx];
  }
  nxt_out[s] = n2;
  dist_out[s] = d;
}

// Grid (ceil(S0 / 256), B), so that no CTA spans two blocks and each loads the C table of its own block.
// dist[s] = D(s) = steps from splitter s to the end of its block's opened cycle (back at rank 0), so the text position of
// splitter s is q0 = (2N_k - 1 - D(s)) mod N_k (splitter 0 = rank 0 = suffix N_k - 1).  Walk len[s] steps: the row at
// step t is the suffix at text position q = q0 + t; its first character F[g] is X_k[n_k-1-q] (q = N_k-1: the sentinel).
// Single-cycle check (DESIGN.md §3.7): L with this eob is the BWT of a text exactly when Psi is one cycle, i.e. when
//   (a) the walk-1 lengths of the block's splitters sum to N_k (every cycle holds a splitter: walk 1 ends on the splitter's
//       own cycle, so the sum counts exactly the rows of cycles that have one), and
//   (b) after the ceil(log2 S0) jump rounds every splitter has nxt == INV_NIL (it lies on the cycle through row 0; on any
//       other cycle a chain never reaches NIL).
// Each CTA adds its part of the sum to chk[k] (chk: [2B] zeroed words; chk[B + k] counts the CTAs of block k that are done)
// and the last CTA of the block compares; a failed test sets bit k of ctrl[CTR_INV_BAD..].  The output is written anyway.
// VERIFY (a forward transform's output): splitters counted from the anchor, F recovered as byte(v) = v - [v > c], and the
// starting points checked — at text position q = N_k - j x (x = floor(N_k / nLF_k), 1 <= j < nLF_k) the row must be
// LFpowers_k[j] (d_eob[256 k + j]); a difference sets bit k like a corrupt block.
template <bool VERIFY>
__global__ void __launch_bounds__(256) k_inv_walk2(const uint32_t* __restrict__ vals, const uint32_t* __restrict__ len,
                                                   const uint32_t* __restrict__ dist, const uint32_t* __restrict__ nxt,
                                                   const uint32_t* __restrict__ C, const InvShape sh, uint8_t* __restrict__ out,
                                                   uint32_t* __restrict__ ctrl, uint32_t* __restrict__ chk) {
  __shared__ uint32_t s_C[258];
  __shared__ uint32_t s_sum, s_open;
  if (ctrl[CTR_ERR]) return;  // (the caller's buffer — possibly the in-place input — stays untouched)
  const uint32_t k = blockIdx.y;
  for (int i = threadIdx.x; i < 258; i += blockDim.x) s_C[i] = C[(size_t)k * 258 + i];
  if (threadIdx.x == 0) { s_sum = 0; s_open = 0; }
  __syncthreads();
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  const bool last = k + 1u == sh.nblocks;
  const bool active = j < (last ? sh.S_last : sh.S0);
  const uint32_t N = last ? sh.N_last : sh.R, n = N - 1u, top = inv_rows(sh) - 1u;
  const uint32_t s = k * sh.S0 + j;
  const uint32_t L = active ? len[s] : 0u;  // (a cycle's splitters split it: the sum never exceeds N_k)
  const uint32_t wsum = __reduce_add_sync(0xFFFFFFFFu, L);
  const bool wopen = __any_sync(0xFFFFFFFFu, active && nxt[s] != INV_NIL);
  if ((threadIdx.x & 31u) == 0u) {
    if (wsum) atomicAdd(&s_sum, wsum);
    if (wopen) s_open = 1u;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicAdd(&chk[k], s_sum);
    if (s_open) inv_mark_bad(ctrl, k);
    __threadfence();
    if (atomicAdd(&chk[sh.nblocks + k], 1u) == gridDim.x - 1u) {  // the last CTA of block k: every part is in chk[k]
      __threadfence();
      if (atomicAdd(&chk[k], 0u) != N) inv_mark_bad(ctrl, k);
    }
  }
  if (!active) return;
  uint8_t* __restrict__ outk = out + (size_t)k * sh.n0;
  const uint32_t base = k * sh.R;
  uint32_t g = base + (VERIFY ? (s_C[sh.eot[k]] - base + j * INV_K) % N : j * INV_K);  // (s_C: block k's C table)
  uint32_t q = (uint32_t)((2ull * N - 1ull - (unsigned long long)dist[s]) % N);
  // VERIFY: the next sampled position is where d = N - q reaches a multiple of x; jj = d / x, rem = d % x, kept per step
  const uint32_t c = VERIFY ? sh.eot[k] : 0u;
  const uint32_t nl = VERIFY ? (last ? sh.nLF_last : sh.nLF) : 1u, x = VERIFY ? N / nl : 1u;
  const uint32_t* __restrict__ LFk = VERIFY ? sh.d_eob + 256u * k : nullptr;
  uint32_t jj = 0, rem = 0;
  bool lf_bad = false;
  if (VERIFY) { jj = (N - q) / x; rem = (N - q) % x; }
  for (uint32_t t = 0; t < L; ++t) {
    if (VERIFY && rem == 0u && jj >= 1u && jj < nl) lf_bad |= g - base != LFk[jj];
    if (q < n) {
      // F[g]: the largest key value v with C[v] <= g (binary search over the 257 bucket starts)
      uint32_t lo = 0, hi = 256;
      while (lo < hi) {
        const uint32_t mid = (lo + hi + 1u) >> 1;
        if (s_C[mid] <= g) lo = mid; else hi = mid - 1u;
      }
      outk[n - 1u - q] = (uint8_t)(VERIFY ? lo - (lo > c ? 1u : 0u) : lo - 1u);
    }
    g = inv_psi(vals, top, g);
    q = (q + 1u == N) ? 0u : q + 1u;
    if (VERIFY) {
      if (q == 0u) { jj = N / x; rem = N % x; }
      else if (rem == 0u) { --jj; rem = x - 1u; }
      else --rem;
    }
  }
  if (VERIFY && lf_bad) inv_mark_bad(ctrl, k);
}

// ---- verification of a forward transform (DESIGN.md §3.10).  Grid (x, B).  Block k restored into rest + k n0 must equal
// X_k, which the forward's text still holds reversed: T'_k = text + k R, X_k[i] = T'_k[n_k - 1 - i].  A difference sets bit k
// of ctrl[CTR_INV_BAD..], like a corrupt block.
__global__ void __launch_bounds__(256) k_inv_verify(const uint8_t* __restrict__ rest, const uint8_t* __restrict__ text,
                                                    const InvShape sh, uint32_t* __restrict__ ctrl) {
  if (ctrl[CTR_ERR]) return;
  const uint32_t k = blockIdx.y;
  const uint32_t n = ((k + 1u == sh.nblocks) ? sh.N_last : sh.R) - 1u;
  const uint8_t* __restrict__ rk = rest + (size_t)k * sh.n0;
  const uint8_t* __restrict__ tk = text + (size_t)k * sh.R;
  bool diff = false;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) diff |= rk[i] != tk[n - 1u - i];
  if (__any_sync(0xFFFFFFFFu, diff) && (threadIdx.x & 31u) == 0u) inv_mark_bad(ctrl, k);
}

// out[i] = text[n - 1 - i]: puts the input of a failed in-place forward transform back from its reversed text.
__global__ void __launch_bounds__(256) k_text_unreverse(const uint8_t* __restrict__ text, uint32_t n, uint8_t* __restrict__ out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = text[n - 1u - i];
}

// Test hook BWTC_DEBUG_CORRUPT_OUT: one byte of the forward output changed before it is verified.
__global__ void k_debug_flip_byte(uint8_t* p) { *p ^= 1u; }
// ... of a raw output: row i, or the next row if i is pidx (= LF[0]; the inverse ignores U[pidx], a change there is no error)
__global__ void k_debug_flip_raw(uint8_t* out, uint32_t i, uint32_t N, const uint32_t* __restrict__ LF) {
  if (LF[0] == i) i = (i + 1u) % N;
  out[i] ^= 1u;
}
// Test hook BWTC_DEBUG_CORRUPT_LF=j: LFpowers[j] of every block that has one changed before the forward output is verified.
__global__ void k_debug_corrupt_lf(uint32_t* LF, uint32_t j, uint32_t nblocks, uint32_t nLF, uint32_t nLF_last) {
  const uint32_t k = threadIdx.x;
  if (k < nblocks && j >= 1u && j < (k + 1u == nblocks ? nLF_last : nLF)) LF[256u * k + j] ^= 1u;
}

// =====================================================================================================
// Run statistics of the transformed block (SURVEY.md §8f row f3; the reference's own TODO at HuffmanCoders.cpp:54:
// "Also gather information about the runs during BWT").  HuffmanEncoder::encodeData re-scans every section of the BWT
// byte by byte to split it into runs (utils::calculateRunFrequenciesAndStoreRuns, Utils.cpp:150-170).  The device has
// the bytes in HBM anyway: two streaming kernels emit the maximal runs of the whole block — (symbol, start position)
// pairs in order — and the host side only slices them at section boundaries.  They are shipped to the host only when
// they are few (a repetitive block: 5 bytes per run instead of a scan over n bytes); for text-like blocks, where three
// out of four positions start a run, the scan on the host stays cheaper than the PCIe traffic.
//   k_run_count : heads per 4096-byte tile (head(i) = i == 0 || out[i] != out[i-1])
//   (k_scan_tile_counts, the forward path's scan, turns them into exclusive offsets)
//   k_run_emit  : symbol[off + k] = out[i], start[off + k] = i for the k-th head of the tile
// =====================================================================================================
constexpr uint32_t RUN_TILE = 4096;  // bytes per CTA (16 per thread)

__device__ __forceinline__ uint32_t run_heads16(const uint8_t* __restrict__ out, uint32_t n, uint32_t i0, uint8_t* b) {
  // 16 consecutive bytes of this thread + the byte before them; returns the head mask
  uint8_t prev = (i0 > 0 && i0 - 1 < n) ? out[i0 - 1] : 0;
  uint32_t mask = 0;
  if (i0 + 16 <= n && (reinterpret_cast<uintptr_t>(out + i0) & 15u) == 0) {
    const uint4 v = *reinterpret_cast<const uint4*>(out + i0);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 16; ++k) b[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
  } else {
#pragma unroll
    for (int k = 0; k < 16; ++k) b[k] = (i0 + k < n) ? out[i0 + k] : 0;
  }
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const uint32_t i = i0 + k;
    if (i < n && (i == 0 || b[k] != prev)) mask |= 1u << k;
    prev = b[k];
  }
  return mask;
}

__global__ void __launch_bounds__(256) k_run_count(const uint8_t* __restrict__ out, uint32_t n, uint32_t* __restrict__ tile_cnt,
                                                   const LadderState* __restrict__ st) {
  __shared__ uint32_t s_w[8];
  if (st->m != 0u) return;  // enqueued speculatively behind the ladder: the block is not finished yet
  uint8_t b[16];
  const uint32_t i0 = blockIdx.x * RUN_TILE + threadIdx.x * 16u;
  uint32_t c = __popc(run_heads16(out, n, i0, b));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int w = 0; w < 8; ++w) t += s_w[w];
    tile_cnt[blockIdx.x] = t;
  }
}

// total[0] = number of runs; the arrays are written only while the index stays below `capacity`.
__global__ void __launch_bounds__(256) k_run_emit(const uint8_t* __restrict__ out, uint32_t n, const uint32_t* __restrict__ tile_cnt,
                                                  const uint32_t* __restrict__ tile_excl, uint32_t ntiles, uint32_t capacity,
                                                  uint8_t* __restrict__ symbol, uint32_t* __restrict__ start,
                                                  uint32_t* __restrict__ total, const LadderState* __restrict__ st) {
  __shared__ uint32_t s_w[8];
  if (st->m != 0u) return;
  uint8_t b[16];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t i0 = blockIdx.x * RUN_TILE + threadIdx.x * 16u;
  const uint32_t mask = run_heads16(out, n, i0, b);
  const uint32_t c = __popc(mask);
  uint32_t inc = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_w[warp] = inc;
  __syncthreads();
  uint32_t woff = 0;
  for (int w = 0; w < warp; ++w) woff += s_w[w];
  uint32_t pos = tile_excl[blockIdx.x] + woff + inc - c;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    if ((mask >> k) & 1u) {
      if (pos < capacity) { symbol[pos] = b[k]; start[pos] = i0 + k; }
      ++pos;
    }
  }
  if (blockIdx.x == ntiles - 1u && threadIdx.x == 0) total[0] = tile_excl[blockIdx.x] + tile_cnt[blockIdx.x];
}

}  // namespace bwtc_b200
