// bwtc_b200/csrc/bwt_kernels.cuh — hand-written sm_100a kernels of the forward-BWT engine.
//
// Algorithm (DESIGN.md §3): suffix array by prefix doubling, never materialised as an array —
// the engine keeps the inverse suffix array rank[] (ISA) and refines it:
//   round 0   : key(i) = first c characters of suffix i as dense b-bit codes (k_pack_round0),
//               LSD radix sort of (key, suffix id [, predecessor code]) with one-sweep digit passes
//               (k_radix_pass), segmented re-rank (k_rerank<ROUND0>): rank[i] = index of i's group head,
//               singletons flagged RANK_DONE and their BWT byte emitted at once.
//   round r>0 : (a) at most 2048 suffixes live: one CTA finishes everything (k_small_rounds);
//               (b) every group <= 128 suffixes: groups are ordered in shared memory without a global sort
//                   (k_seg_round + k_apply_ranks) from the rank-ordered live lists k_rerank staged;
//               (c) otherwise a packed (rank[i] >> 1, rank[i+h] + 1) 64-bit key for every still-live suffix
//                   (k_build_keys in text order, or k_build_from_list), same radix sort, k_rerank<false>.
//   final     : pidx / LFpowers extraction and the bwtc hole-fill (k_finish); the BWT bytes were written by the
//               re-rank kernels (emit_bwt) the moment each suffix became unique.
//   batches   : runs of small equal-sized blocks are one text with the block number on top of every key and a
//               reserved sentinel code (k_prep_batch, k_finish_batch; DESIGN.md §3.6).
// All of this replaces sort_typeBstar + sssort + trsort + construct_BWT of the reference
// (bwtransforms/divsufsort.c:38-192,328-404; sssort.c:746-815; trsort.c:554-586) — it is NOT a port of
// them: no B*-suffix classification, no induced sorting, no introsort.
//
// Everything is integer / byte work bound by HBM bandwidth; no tensor cores are used on purpose.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bwtc_b200 {

constexpr uint32_t RANK_DONE = 0x80000000u;  // bit 31 of rank[i]: suffix i is alone in its group (final)
constexpr uint32_t RANK_MASK = 0x7FFFFFFFu;

// ---- control words (one uint32 array per context).  Words [0, CTR_STICKY) are zeroed once per block, the others by
//      a memset at the start of every sort round.
constexpr int CTR_ERR = 0;         // != 0: a look-back watchdog fired / an internal check failed.  STICKY: every later
                                   // kernel of the block returns at entry, so nothing consumes half-written buffers
constexpr int CTR_STICKY = 8;
constexpr int CTR_PASS0 = 8;       // [8..23]  tile ticket counters of the radix passes (ticket mode only)
constexpr uint32_t CTR_STATIC = 0xFFFFFFFFu;      // "no ticket counter: tile id = blockIdx.x"
constexpr uint32_t CTR_STATIC_REV = 0xFFFFFFFEu;  // test hook: tile id = gridDim.x - 1 - blockIdx.x (a dispatch order
                                                  // that is as wrong as it can be; see tests/test_gpu_parity.py)
constexpr int CTR_CURSOR = 24;     // output cursor of k_build_keys (== number of live records emitted)
constexpr int CTR_LIVE = 25;       // records still in non-singleton groups after the re-rank of this round
constexpr int CTR_MAXGROUP = 26;   // size of the largest non-singleton group seen by the re-rank of this round
constexpr int CTR_UPD = 27;        // cursor of the rank-update list written by k_seg_round
constexpr int CTR_RERANK = 32;     // [32..47] tile ticket counters of the k_rerank window launches (ticket mode only)
constexpr int MAX_RERANK_WINDOWS = 16;
constexpr int CTR_WORDS = 64;

// look-back status words of the radix pass: bit 31 = "inclusive prefix" (else: this tile's count only), bits 30..0 =
// count + 1, so an unpublished word is simply 0 and counts up to 2^31 - 2 fit — the reference's block limit
// (Compressor.cpp:78-79) — without a second flag bit.
constexpr uint32_t LB_PREFIX = 0x80000000u, LB_VALUE = 0x7FFFFFFFu;
constexpr uint32_t LB_PAD_WORD = LB_PREFIX | 1u;  // "inclusive prefix 0": what the pad rows in front of tile 0 hold
// Spin watchdog of the look-back loops (a violated dispatch-order assumption becomes an error, not a hang).
// __constant__ so a test can shrink it (BWTC_DEBUG_SPIN_LIMIT, read by bwtc_cuda_ctx_create).
__constant__ uint32_t g_lb_spin_limit = 1u << 24;
constexpr int LB_PAD_ROWS = 8;  // rows of "prefix 0" in front of tile 0 (>= LB_BATCH): look-back loads need no bounds check
#ifndef BWTC_LB_BATCH
#define BWTC_LB_BATCH 8
#endif
// Predecessor status words fetched per look-back round trip.  With T tiles in flight staggered by dt cycles
// and a round trip of RT cycles the look-back settles at L = RT / (1 - RT / (dt * BATCH)): the batch must
// satisfy dt * BATCH >> RT or the walk chases an ever longer chain of aggregate-only predecessors.
constexpr int LB_BATCH = BWTC_LB_BATCH;
#ifndef BWTC_LB_BATCH9
#define BWTC_LB_BATCH9 2
#endif
constexpr int LB_BATCH9 = BWTC_LB_BATCH9;  // per digit in the 9-bit pass (two digits per thread); measured 2/4/6/8: 1.894/1.905/1.935/1.990 ms per sort
static_assert(LB_BATCH9 <= LB_PAD_ROWS, "the look-back batch must not read past the pad rows");
static_assert(LB_BATCH <= LB_PAD_ROWS, "the look-back batch must not read past the pad rows");

// Record streams of k_radix_pass: plain loads, streaming (evict-first) stores.  Measured on the 32 MiB Markov block:
// .cs stores -1.9% sort time, .cg stores the same, .cs loads +1.6% (profiles/r01_experiments.md).
#define BWTC_LD(p) (*(p))
#define BWTC_ST(p, v) __stcs(p, v)

#ifndef BWTC_RS_BLOCK
#define BWTC_RS_BLOCK 256
#endif
#ifndef BWTC_RS_MINB
#define BWTC_RS_MINB 3
#endif
#ifndef BWTC_RS_MINB32
#define BWTC_RS_MINB32 4
#endif
#ifndef BWTC_RS_IPT64
#define BWTC_RS_IPT64 16
#endif
#ifndef BWTC_RS_IPT32
#define BWTC_RS_IPT32 16
#endif

__device__ __forceinline__ uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_volatile_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_volatile_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Lanes of the warp whose 8-bit digit equals mine (8 ballots; the multi-split primitive of the sort).
// Inline PTX pins 3 instructions per bit (ballot + one of two predicated LOP3s; the 8 bit-test predicates come
// from a single R2P); the C++ "bit ? bal : ~bal" form compiled to 6 per bit.
__device__ __forceinline__ uint32_t match_digit8(uint32_t d) {
  uint32_t m = 0xFFFFFFFFu;
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b32 t;\n"
        "and.b32 t, %1, %2;\n"
        "setp.ne.u32 p, t, 0;\n"
        "vote.sync.ballot.b32 t, p, 0xffffffff;\n"
        "@p and.b32 %0, %0, t;\n"
        "@!p lop3.b32 %0, %0, t, 0, 0x30;\n"  // m & ~t in one LOP3
        "}\n"
        : "+r"(m)
        : "r"(d), "r"(1u << b));
  }
  return m;
}

// The same with 9 ballots (9-bit digits, BWTC radix-9 passes).
__device__ __forceinline__ uint32_t match_digit9(uint32_t d) {
  uint32_t m = 0xFFFFFFFFu;
#pragma unroll
  for (int b = 0; b < 9; ++b) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b32 t;\n"
        "and.b32 t, %1, %2;\n"
        "setp.ne.u32 p, t, 0;\n"
        "vote.sync.ballot.b32 t, p, 0xffffffff;\n"
        "@p and.b32 %0, %0, t;\n"
        "@!p lop3.b32 %0, %0, t, 0, 0x30;\n"
        "}\n"
        : "+r"(m)
        : "r"(d), "r"(1u << b));
  }
  return m;
}

// Exclusive sum-scan over the first 256 threads of the CTA (value of threads >= 256 is ignored).
// Every thread of the CTA must call it (contains __syncthreads). s_tot: 8 words of shared memory.
__device__ __forceinline__ uint32_t scan256_excl(uint32_t v, uint32_t* s_tot) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
    if (lane >= o) inc += t;
  }
  if (w < 8 && lane == 31) s_tot[w] = inc;
  __syncthreads();
  uint32_t base = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint32_t t = s_tot[i];
    if (i < w) base += t;
  }
  __syncthreads();
  return base + inc - v;
}

// Two exclusive sum-scans over the 256 threads of the CTA at once (same barriers); tot0 / tot1 receive the totals.
// s_tot: 16 words of shared memory.
__device__ __forceinline__ void scan256_excl2(uint32_t v0, uint32_t v1, uint32_t* s_tot, uint32_t& e0, uint32_t& e1,
                                              uint32_t& tot0, uint32_t& tot1) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  uint32_t i0 = v0, i1 = v1;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t0 = __shfl_up_sync(0xFFFFFFFFu, i0, o);
    const uint32_t t1 = __shfl_up_sync(0xFFFFFFFFu, i1, o);
    if (lane >= o) { i0 += t0; i1 += t1; }
  }
  if (w < 8 && lane == 31) { s_tot[w] = i0; s_tot[8 + w] = i1; }
  __syncthreads();
  uint32_t b0 = 0, b1 = 0, a0 = 0, a1 = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint32_t t0 = s_tot[i], t1 = s_tot[8 + i];
    a0 += t0; a1 += t1;
    if (i < w) { b0 += t0; b1 += t1; }
  }
  __syncthreads();
  e0 = b0 + i0 - v0;
  e1 = b1 + i1 - v1;
  tot0 = a0;
  tot1 = a1;
}

// =====================================================================================================
// k_prep_block — block contract front end.  Replaces std::reverse + "*end = 0" of
// BWTransform::doTransform(BWTBlock&,freqs) (BWTransform.cpp:53-55) and the ++freqs[U[i]] loop of
// divbwtf (divsufsort.c:506-512): text[i] = X[n-1-i], text[n] = 0 (+ zero padding), hist = byte counts.
// One thread produces 4 text bytes (coalesced 32-bit stores; the reversed byte loads hit L1).
// =====================================================================================================
__global__ void __launch_bounds__(256) k_prep_block(const uint8_t* __restrict__ X, uint32_t n,
                                                    uint8_t* __restrict__ text, uint32_t padded_words,
                                                    uint32_t* __restrict__ hist) {
  __shared__ uint32_t s_hist[256];
  s_hist[threadIdx.x] = 0;
  __syncthreads();
  for (uint32_t wi = blockIdx.x * blockDim.x + threadIdx.x; wi < padded_words; wi += gridDim.x * blockDim.x) {
    const uint32_t o = wi * 4u;
    uint32_t packed = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t i = o + j;
      if (i < n) {
        const uint32_t ch = X[n - 1u - i];
        packed |= ch << (8 * j);
        atomicAdd(&s_hist[ch], 1u);
      }
    }
    reinterpret_cast<uint32_t*>(text)[wi] = packed;
  }
  __syncthreads();
  const uint32_t v = s_hist[threadIdx.x];
  if (v) atomicAdd(&hist[threadIdx.x], v);
}

// k_hist_bytes — raw contract front end: hist of T[0..cnt) (the freqs of divbwtf, divsufsort.c:506-512).
__global__ void __launch_bounds__(256) k_hist_bytes(const uint8_t* __restrict__ T, uint32_t cnt,
                                                    uint32_t* __restrict__ hist) {
  __shared__ uint32_t s_hist[256];
  s_hist[threadIdx.x] = 0;
  __syncthreads();
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += gridDim.x * blockDim.x)
    atomicAdd(&s_hist[T[i]], 1u);
  __syncthreads();
  const uint32_t v = s_hist[threadIdx.x];
  if (v) atomicAdd(&hist[threadIdx.x], v);
}

// k_prep_batch — front end for a batch of small blocks sorted as one text (DESIGN.md §3.6).  Block k (bytes
// srcs[k][0..n_k)) becomes text[k*stride .. k*stride + n_k] = reverse(X_k) . 0x00 with stride = n_0 + 1; all blocks
// have n_0 bytes except the last (n_last <= n_0).  hist[k][256] = byte counts of block k (its freqs).
// grid = (x, nblocks): every CTA writes a share of the text words and counts a share of its own block.
__global__ void __launch_bounds__(256) k_prep_batch(const uint8_t* const* __restrict__ srcs, uint32_t n0, uint32_t n_last,
                                                    uint32_t nblocks, uint8_t* __restrict__ text, uint32_t Ntot,
                                                    uint32_t padded_words, uint32_t* __restrict__ hist) {
  __shared__ uint32_t s_hist[256];
  s_hist[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t stride = n0 + 1u;
  const uint32_t cta = blockIdx.y * gridDim.x + blockIdx.x, nctas = gridDim.x * gridDim.y;
  for (uint32_t wi = cta * blockDim.x + threadIdx.x; wi < padded_words; wi += nctas * blockDim.x) {
    uint32_t packed = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t p = wi * 4u + j;
      if (p < Ntot) {
        const uint32_t k = p / stride, i = p - k * stride;
        const uint32_t nk = (k + 1u == nblocks) ? n_last : n0;
        if (i < nk) packed |= (uint32_t)srcs[k][nk - 1u - i] << (8 * j);
      }
    }
    reinterpret_cast<uint32_t*>(text)[wi] = packed;
  }
  const uint32_t k = blockIdx.y;
  const uint32_t nk = (k + 1u == nblocks) ? n_last : n0;
  const uint8_t* X = srcs[k];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nk; i += gridDim.x * blockDim.x)
    atomicAdd(&s_hist[X[i]], 1u);
  __syncthreads();
  const uint32_t v = s_hist[threadIdx.x];
  if (v) atomicAdd(&hist[k * 256u + threadIdx.x], v);
}

// =====================================================================================================
// k_window_sample / k_window_pairs — policy input for the round-0 key shape (DESIGN.md §3.2).  ~2^16 strided
// 8-byte windows of the block are inserted into an open-addressing table (atomicCAS on the window itself, a
// counter per slot); the second kernel reduces sum m(m-1)/2 = number of colliding sample pairs.  The host
// compares that MEASURED 8-gram collision rate with what an i.i.d. source with the block's byte histogram
// would give: text and repeats exceed it by orders of magnitude, random bytes and DNA match it.  No source
// model is assumed beyond that comparison.
// =====================================================================================================
constexpr uint32_t WS_SLOTS = 1u << 17;
constexpr unsigned long long WS_EMPTY = ~0ull;

__global__ void __launch_bounds__(256) k_window_sample(const uint8_t* __restrict__ X, uint32_t n, uint32_t stride,
                                                       uint32_t nsamp, unsigned long long* __restrict__ tab_key,
                                                       uint32_t* __restrict__ tab_cnt) {
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < nsamp; s += gridDim.x * blockDim.x) {
    const uint32_t i = s * stride;  // i + 8 <= n guaranteed by the host
    unsigned long long key = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) key = (key << 8) | (unsigned long long)X[i + k];
    if (key == WS_EMPTY) key = WS_EMPTY - 1;
    unsigned long long hsh = key * 0x9E3779B97F4A7C15ull;
    uint32_t slot = (uint32_t)(hsh >> 40) & (WS_SLOTS - 1);
    for (int probe = 0; probe < 64; ++probe) {
      const unsigned long long prev = atomicCAS(&tab_key[slot], WS_EMPTY, key);
      if (prev == WS_EMPTY || prev == key) {
        atomicAdd(&tab_cnt[slot], 1u);
        break;
      }
      slot = (slot + 1) & (WS_SLOTS - 1);
    }
  }
}

__global__ void __launch_bounds__(1024) k_window_pairs(const uint32_t* __restrict__ tab_cnt, double* __restrict__ out) {
  __shared__ double s_a[32], s_b[32];
  double pairs = 0.0, tot = 0.0;
  for (uint32_t i = threadIdx.x; i < WS_SLOTS; i += 1024) {
    const double m = (double)tab_cnt[i];
    pairs += m * (m - 1.0) * 0.5;
    tot += m;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    pairs += __shfl_down_sync(0xFFFFFFFFu, pairs, o);
    tot += __shfl_down_sync(0xFFFFFFFFu, tot, o);
  }
  if ((threadIdx.x & 31) == 0) { s_a[threadIdx.x >> 5] = pairs; s_b[threadIdx.x >> 5] = tot; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, bb = 0;
    for (int w = 0; w < 32; ++w) { a += s_a[w]; bb += s_b[w]; }
    out[0] = a;   // colliding sample pairs
    out[1] = bb;  // samples inserted
  }
}

// =====================================================================================================
// k_pack_round0 — round-0 keys.  Position t of the key array holds suffix i = N-1-t (descending suffix
// ids, see DESIGN.md §3.2: with a stable sort, suffixes whose c-character window runs past the end of
// the text then precede every other suffix with an equal key, which is their correct order), so no code
// point has to be reserved for the sentinel.  key = c dense b-bit codes, most significant = first char.
// The digit histograms of the radix passes of the round are accumulated here (shared-memory atomics, one
// global flush per CTA; persistent grid) — one representative digit per phase class, the others are derived
// by k_hist_derive — so the sort never re-reads the keys to count.
// Replaces the bucket counting of sort_typeBstar (divsufsort.c:62-74).
// =====================================================================================================
struct PackParams {
  uint8_t lut[256];   // byte -> dense code
  uint32_t bits;      // b
  uint32_t chars;     // c  (c*b + rbits <= 8*sizeof(KeyT), c <= 64)
  // Spare low key bits (the last digit pass runs anyway) hold the TOP rbits bits of the code of character c+1: a monotone
  // coarsening of that character, so key order still implies suffix order and equal keys still share c characters — the
  // doubling distance stays c, but round 0 leaves fewer suffixes tied (Markov 32 MiB: 7.7% -> 3.0% with 4 of 6 bits).
  uint32_t rbits;     // 0 <= rbits < b; 0 in batch mode
  // batch of nblocks > 1 blocks (text = concatenation, block k at k*stride): code 0 is RESERVED for the sentinel
  // positions (lut[] >= 1 for every data byte), and the block number is stored above the c characters
  uint32_t nblocks;
  uint32_t stride;
};

constexpr int GRAM_BITS = 12;  // gram mode of k_pack_round0 / k_hist_from_gram (see GramParams)

template <typename KeyT>
__global__ void __launch_bounds__(256) k_pack_round0(const uint8_t* __restrict__ text, uint32_t N,
                                                     KeyT* __restrict__ keys, PackParams pp,
                                                     uint32_t* __restrict__ hist, uint32_t hist_mask, uint32_t ntiles,
                                                     uint32_t rb, uint32_t* __restrict__ gram) {
  // rb: digit width of the sort that follows (8 or 9); digit p = (key >> rb*p) & (2^rb - 1), histogram p at hist + p * 2^rb
  // gram != nullptr (hist_mask == 0): instead of digit histograms, ONE histogram of the low GRAM_BITS bits of every key —
  // the last 2 (6-bit codes) or 4 (3-bit codes) characters of its window; every digit histogram is a projection of it
  // (k_hist_from_gram).  One shared-memory atomic per key into 4096 bins instead of four into 256-bin histograms.
  constexpr int BLOCK = 256, IPT = 8, TILE = BLOCK * IPT;
  __shared__ uint8_t s_lut[256];
  __shared__ uint8_t s_code[TILE + 64];
  __shared__ uint32_t s_hist[8 * 512];  // digit histograms, or the gram histogram (1 << GRAM_BITS bins)
  static_assert((1 << GRAM_BITS) <= 8 * 512, "the gram histogram shares the digit histograms' shared memory");
  const int tid = threadIdx.x;
  const uint32_t dmask = (1u << rb) - 1u;
  s_lut[tid] = pp.lut[tid];
#pragma unroll
  for (int p = 0; p < 16; ++p) s_hist[p * 256 + tid] = 0;
  __syncthreads();
  const uint32_t c = pp.chars, b = pp.bits;
  for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const uint32_t t0 = tile * (uint32_t)TILE;
    const long long wlo = (long long)N - (long long)t0 - TILE;  // text index held in s_code[0]
    for (int q = tid; q < TILE + 64; q += BLOCK) {
      const long long g = wlo + q;
      s_code[q] = (g >= 0 && g < (long long)N) ? s_lut[text[g]] : (uint8_t)0;
    }
    if (pp.nblocks > 1u) {
      // the sentinel of block k sits at (k+1)*stride - 1 (the last block's at N-1): it is the reserved code 0,
      // whatever lut[] says about a 0x00 data byte
      __syncthreads();
      const long long lo = wlo < 0 ? 0 : wlo;
      for (long long k = lo / pp.stride + tid;; k += BLOCK) {
        long long sp = (k + 1) * (long long)pp.stride - 1;
        if (sp >= (long long)N) sp = (long long)N - 1;
        if (sp - wlo >= TILE + 63) break;
        if (sp >= wlo) s_code[sp - wlo] = 0;
        if (sp == (long long)N - 1) break;
      }
    }
    __syncthreads();
    // Thread-blocked: 8 consecutive positions per thread.  Position t holds suffix N-1-t, so walking t upwards
    // walks the text downwards and each key is the previous one shifted by one character plus one new code:
    //   key(i) = code(T[i]) << (c-1)b | key(i+1) >> b        (1 shared-memory byte per key instead of c)
    {
      const uint32_t u0 = (uint32_t)tid * IPT;
      const int q0 = TILE - 1 - (int)u0;  // s_code index of the first character of the thread's first suffix
      KeyT key = 0;
      for (uint32_t j = 0; j < c; ++j) key = (KeyT)(key << b) | (KeyT)s_code[q0 + j];
      const uint32_t topshift = (c - 1) * b;
      const uint32_t rbits = pp.rbits;
      KeyT out[IPT];
#pragma unroll
      for (int k = 0; k < IPT; ++k) {
        if (k > 0) key = (KeyT)((KeyT)s_code[q0 - k] << topshift) | (KeyT)(key >> b);
        out[k] = key;
        // (c <= 63 when rbits > 0, so q0 - k + c <= TILE + 62 is inside the loaded window)
        if (rbits) out[k] = (KeyT)(key << rbits) | (KeyT)((uint32_t)s_code[q0 - k + (int)c] >> (b - rbits));
      }
      if (pp.nblocks > 1u) {  // block number above the characters: suffix of position t0+u0+k is N-1-(t0+u0+k)
        const uint32_t blkshift = c * b;
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
          const uint32_t t = t0 + u0 + (uint32_t)k;
          if (t < N) out[k] |= (KeyT)((N - 1u - t) / pp.stride) << blkshift;
        }
      }
      const uint32_t t = t0 + u0;
      if (t + IPT <= N) {
        if (sizeof(KeyT) == 8) {
          ulonglong2* dst = reinterpret_cast<ulonglong2*>(keys + t);  // t % 8 == 0, keys 256-byte aligned
#pragma unroll
          for (int k = 0; k < IPT; k += 2) dst[k / 2] = make_ulonglong2((unsigned long long)out[k], (unsigned long long)out[k + 1]);
        } else {
          uint4* dst = reinterpret_cast<uint4*>(keys + t);
#pragma unroll
          for (int k = 0; k < IPT; k += 4)
            dst[k / 4] = make_uint4((uint32_t)out[k], (uint32_t)out[k + 1], (uint32_t)out[k + 2], (uint32_t)out[k + 3]);
        }
      } else {
#pragma unroll
        for (int k = 0; k < IPT; ++k)
          if (t + k < N) keys[t + k] = out[k];
      }
      if (gram) {
#pragma unroll
        for (int k = 0; k < IPT; ++k)
          if (t + k < N) atomicAdd(&s_hist[(uint32_t)(out[k] >> pp.rbits) & ((1u << GRAM_BITS) - 1u)], 1u);
      } else {
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
          if (t + k < N) {
#pragma unroll
            for (int p = 0; p < (int)(sizeof(KeyT)); ++p)
              if ((hist_mask >> p) & 1u) atomicAdd(&s_hist[(p << rb) + ((uint32_t)(out[k] >> (rb * p)) & dmask)], 1u);
          }
        }
      }
    }
    __syncthreads();
  }
  if (gram) {
    for (uint32_t e = tid; e < (1u << GRAM_BITS); e += BLOCK) {
      const uint32_t v = s_hist[e];
      if (v) atomicAdd(&gram[e], v);
    }
    return;
  }
#pragma unroll
  for (int p = 0; p < (int)(sizeof(KeyT)); ++p) {
    if (!((hist_mask >> p) & 1u)) continue;
    for (uint32_t e = tid; e <= dmask; e += BLOCK) {
      const uint32_t v = s_hist[(p << rb) + e];
      if (v) atomicAdd(&hist[(p << rb) + e], v);
    }
  }
}

// =====================================================================================================
// k_hist_derive — the digit histograms of a sliding-window key are shifts of each other.  Digit p of key(i)
// depends only on the characters i+j_lo(p).. and on the phase (8p mod b) at which the 8-bit digit cuts the b-bit
// codes; two digits p > r of equal phase satisfy  digit_p(key(i)) == digit_r(key(i - t)),  t = 8(p-r)/b.  So
//   H_p = H_r - sum_{i=N-t}^{N-1} e(digit_r(key(i))) + sum_{i=0}^{t-1} e(digit_p(key(i)))
// and k_pack_round0 only has to count one representative digit per phase class with shared-memory atomics
// (its most expensive part): 3 of 8 digits for 6-bit codes, 1 of 4 for bytes and DNA.  Block q of the grid
// derives digit derive_p[q] from representative derive_r[q].
// =====================================================================================================
struct DeriveParams {
  uint32_t count;
  uint8_t p[8], r[8], t[8];
};

// Gram mode (6-bit and 3-bit codes): G[g] = number of suffixes whose key has g in its low GRAM_BITS bits = its last W
// characters (W * b = 12).  Digit p of key(i) lies inside the W characters that start u_p characters above the key's low
// end, and those are the LAST W characters of key(i - u_p) — the window slid by u_p positions, zero padding included, since
// padding depends on the text position only.  So
//   H_p[d] = sum_g G[g] [(g >> s_p) & dmask == d]  -  sum_{i = N-u_p}^{N-1} e((low12(key(i)) >> s_p) & dmask)   (no partner)
//                                                  +  sum_{i = 0}^{u_p - 1} e(digit_p(key(i)))                    (not covered)
// with 8p (or 9p) = b u_p + s_p, u_p capped so the W characters stay inside the key.  Block p of the grid builds H_p.
// With partial bits (PackParams::rbits) everything above is in the coordinates of E = key >> rbits, the c exact characters:
// G counts the low 12 bits of E, digit p is E bits [rb p - rbits, ...).  The lowest digit then reaches below E into the
// partial character: its 12-bit window is the low window of E(i + 1) (u = -1, flag below) and
//   H_0 = projection(G) - e(window of suffix 0) + e(window of the all-padding "suffix N" = 0).
struct GramParams {
  uint32_t npass;
  uint8_t u[8], s[8];
  uint8_t next[8];  // 1: u = -1 (the window of the following suffix)
};

template <typename KeyT>
__device__ __forceinline__ KeyT pack_key_at(const uint8_t* __restrict__ text, uint32_t N, uint32_t i, const uint8_t* lut,
                                            uint32_t b, uint32_t c, uint32_t rbits) {
  KeyT key = 0;
  for (uint32_t j = 0; j < c; ++j) {
    const uint32_t g = i + j;
    key = (KeyT)(key << b) | (KeyT)((g < N) ? lut[text[g]] : 0u);
  }
  if (rbits) {
    const uint32_t g = i + c;
    key = (KeyT)(key << rbits) | (KeyT)(((g < N) ? (uint32_t)lut[text[g]] : 0u) >> (b - rbits));
  }
  return key;
}

template <typename KeyT>
__global__ void __launch_bounds__(256) k_hist_derive(const uint8_t* __restrict__ text, uint32_t N, PackParams pp,
                                                     DeriveParams dp, uint32_t* __restrict__ hist, uint32_t rb) {
  __shared__ uint8_t s_lut[256];
  __shared__ uint32_t s_h[512];
  const int tid = threadIdx.x;
  const uint32_t p = dp.p[blockIdx.x], r = dp.r[blockIdx.x], t = dp.t[blockIdx.x];
  const uint32_t dmask = (1u << rb) - 1u;
  s_lut[tid] = pp.lut[tid];
  for (uint32_t e = tid; e <= dmask; e += 256) s_h[e] = hist[(r << rb) + e];
  __syncthreads();
  if ((uint32_t)tid < t) {
    if ((uint32_t)tid < N) {  // head term: suffix i = tid counted for digit p
      const KeyT kh = pack_key_at<KeyT>(text, N, (uint32_t)tid, s_lut, pp.bits, pp.chars, pp.rbits);
      atomicAdd(&s_h[(uint32_t)(kh >> (rb * p)) & dmask], 1u);
    }
    if ((uint32_t)tid < N) {  // tail term: suffix i = N-1-tid was counted for digit r but has no partner
      const KeyT kt = pack_key_at<KeyT>(text, N, N - 1u - (uint32_t)tid, s_lut, pp.bits, pp.chars, pp.rbits);
      atomicSub(&s_h[(uint32_t)(kt >> (rb * r)) & dmask], 1u);
    }
  }
  __syncthreads();
  for (uint32_t e = tid; e <= dmask; e += 256) hist[(p << rb) + e] = s_h[e];
}

template <typename KeyT>
__global__ void __launch_bounds__(256) k_hist_from_gram(const uint8_t* __restrict__ text, uint32_t N, PackParams pp,
                                                        GramParams gp, const uint32_t* __restrict__ gram,
                                                        uint32_t* __restrict__ hist, uint32_t rb) {
  __shared__ uint8_t s_lut[256];
  __shared__ uint32_t s_h[512];
  const int tid = threadIdx.x;
  const uint32_t p = blockIdx.x, u = gp.u[p], sh = gp.s[p];
  const uint32_t dmask = (1u << rb) - 1u;
  s_lut[tid] = pp.lut[tid];
  s_h[tid] = 0;
  s_h[tid + 256] = 0;
  __syncthreads();
  for (uint32_t g = tid; g < (1u << GRAM_BITS); g += 256) {
    const uint32_t v = gram[g];
    if (v) atomicAdd(&s_h[(g >> sh) & dmask], v);
  }
  if (gp.next[p]) {
    if (tid == 0) {
      const KeyT k0 = pack_key_at<KeyT>(text, N, 0u, s_lut, pp.bits, pp.chars, pp.rbits);
      atomicSub(&s_h[(((uint32_t)(k0 >> pp.rbits) & ((1u << GRAM_BITS) - 1u)) >> sh) & dmask], 1u);
      atomicAdd(&s_h[0], 1u);
    }
  } else if ((uint32_t)tid < u && (uint32_t)tid < N) {
    const KeyT kh = pack_key_at<KeyT>(text, N, (uint32_t)tid, s_lut, pp.bits, pp.chars, pp.rbits);  // head: suffix tid, digit p directly
    atomicAdd(&s_h[(uint32_t)(kh >> (rb * p)) & dmask], 1u);
    const KeyT kt = pack_key_at<KeyT>(text, N, N - 1u - (uint32_t)tid, s_lut, pp.bits, pp.chars, pp.rbits);  // tail: counted, no partner
    atomicSub(&s_h[(((uint32_t)(kt >> pp.rbits) & ((1u << GRAM_BITS) - 1u)) >> sh) & dmask], 1u);
  }
  __syncthreads();
  for (uint32_t e = tid; e <= dmask; e += 256) hist[(p << rb) + e] = s_h[e];
}

// =====================================================================================================
// k_build_keys — doubling round r >= 1.  Text-order scan of rank[]: both reads (rank[i], rank[i+h]) are
// coalesced; only suffixes still in a non-singleton group emit a record.  key = rank[i] << lo_bits |
// (rank[i+h] + 1), 0 in the low part when i+h is past the end (sorts first = "shorter suffix first").
// Compaction is fused (warp ballots -> CTA offsets -> ONE global atomic per tile; record order is
// irrelevant to the sort) and so are the digit histograms of every pass of this round.
// Replaces "ISAd = ISA + depth" + tr_introsort's key access of trsort (trsort.c:327-552,563).
// =====================================================================================================
__global__ void __launch_bounds__(256) k_build_keys(const uint32_t* __restrict__ rank, uint32_t N, uint32_t h,
                                                    int lo_bits, unsigned long long* __restrict__ keys,
                                                    uint32_t* __restrict__ idx, uint32_t* __restrict__ ctrl,
                                                    uint32_t* __restrict__ hist, int npass, uint32_t ntiles,
                                                    uint32_t rb) {
  constexpr int BLOCK = 256, IPT = 8, TILE = BLOCK * IPT, WARPS = BLOCK / 32;
  __shared__ uint32_t s_hist[8 * 512];
  __shared__ uint32_t s_wtot[WARPS];
  __shared__ uint32_t s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t dmask = (1u << rb) - 1u;
  if (ctrl[CTR_ERR]) return;
#pragma unroll
  for (int p = 0; p < 16; ++p) s_hist[p * 256 + tid] = 0;
  __syncthreads();
  for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    // thread-blocked: 8 consecutive suffixes per thread, two 128-bit loads issued back to back (rank[] is
    // 256-byte aligned and padded, so the vector loads of the last tile stay in bounds)
    const uint32_t i0 = tile * (uint32_t)TILE + tid * IPT;
    uint32_t r[IPT];
    {
      const uint4* pr = reinterpret_cast<const uint4*>(rank + i0);
      uint4 a = make_uint4(RANK_DONE, RANK_DONE, RANK_DONE, RANK_DONE), b4 = a;
      if (i0 < N) a = pr[0];
      if (i0 + 4 < N) b4 = pr[1];
      r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w;
      r[4] = b4.x; r[5] = b4.y; r[6] = b4.z; r[7] = b4.w;
    }
    uint32_t livemask = 0;
#pragma unroll
    for (int k = 0; k < IPT; ++k)
      if (i0 + k < N && !(r[k] & RANK_DONE)) livemask |= 1u << k;
    // second key halves: independent gathers, only for live suffixes
    uint32_t r2[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      r2[k] = 0;
      if ((livemask >> k) & 1u) {
        const uint32_t i = i0 + k;
        if (h < N - i) r2[k] = (rank[i + h] & RANK_MASK) + 1u;
      }
    }
    // CTA-wide exclusive scan of the per-thread live counts -> one global atomic per tile
    const uint32_t cnt = __popc(livemask);
    uint32_t inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) s_wtot[warp] = inc;
    __syncthreads();
    uint32_t woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) {
      const uint32_t t = s_wtot[w];
      if (w < warp) woff += t;
      total += t;
    }
    if (tid == 0) s_base = total ? atomicAdd(&ctrl[CTR_CURSOR], total) : 0u;
    __syncthreads();
    uint32_t pos = s_base + woff + inc - cnt;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      if ((livemask >> k) & 1u) {
        // high part = rank >> 1: a live group has >= 2 members, so the heads of two live groups differ by >= 2 and
        // rank >> 1 still identifies (and orders) the group; the dropped bit rides in bit 31 of the id payload
        // (ids are < 2^31).  One bit less per key is one digit pass less per round at N = 2^k + 1.
        const unsigned long long key = ((unsigned long long)(r[k] >> 1) << lo_bits) | (unsigned long long)r2[k];
        keys[pos] = key;
        idx[pos] = (i0 + k) | ((r[k] & 1u) << 31);
        ++pos;
        for (int p = 0; p < npass; ++p) atomicAdd(&s_hist[(p << rb) + ((uint32_t)(key >> (rb * p)) & dmask)], 1u);
      }
    }
  }
  __syncthreads();
  for (int p = 0; p < npass; ++p)
    for (uint32_t e = tid; e <= dmask; e += BLOCK) {
      const uint32_t v = s_hist[(p << rb) + e];
      if (v) atomicAdd(&hist[(p << rb) + e], v);
    }
}

// =====================================================================================================
// k_radix_pass — one 8-bit digit pass of the LSD radix sort over (key, suffix id) records, single sweep:
//   * tile id = block index (CTAs are dispatched in index order, so a tile only ever waits on tiles that already
//     started); atomic tickets only in the watchdog-fallback mode,
//   * warp-striped coalesced loads, keys/values held in registers,
//   * per-warp digit ranking with 8 ballots per item (match_digit8) into per-warp shared histograms,
//   * per-digit decoupled look-back across tiles (status word = 2 flag bits + 30-bit count; the data
//     travels inside the flag word, so no fence is needed), with a spin watchdog instead of a hang,
//   * records are staged in shared memory in sorted order and written out with consecutive threads
//     writing consecutive addresses of a bin's run (coalesced scatter, streaming stores).
// HBM traffic per record: read key+id, write key+id — the algorithmic minimum for an out-of-place pass.
// IOTA: first pass of round 0 — suffix ids are implied by position (id = iota_top - position), not read.
// Stable, which the round-0 sentinel handling relies on.
// Replaces sssort/trsort's comparison sorting (sssort.c:310,654,746; trsort.c:327).
// =====================================================================================================
#ifdef BWTC_PROFILE_STAGES
__device__ unsigned long long* g_prof_buf = nullptr;  // [tiles][16] SM-clock stamps (profiling builds only)
#define BWTC_PROF(k) do { if (threadIdx.x == 0 && g_prof_buf) g_prof_buf[(size_t)tile * 16 + (k)] = clock64(); } while (0)
#else
#define BWTC_PROF(k) do { } while (0)
#endif

template <typename KeyT, int BLOCK, int IPT, bool AUX = false, int RB = 8>
struct RadixPassSmem {
  static constexpr int TILE = BLOCK * IPT;
  static constexpr int WARPS = BLOCK / 32;
  static constexpr size_t bytes =
      (sizeof(KeyT) + 4) * TILE + sizeof(uint32_t) * (WARPS * 256 + (1 << RB) + 32) + (AUX ? TILE : 0);
};

// AUX: a third, one-byte payload travels with every record — the dense code of the character preceding the
// suffix, for blocks whose id has no spare bits for it (pack_bits) and whose text is too large for an L2-resident
// gather at emission time.  The IOTA pass produces it (top character of the next key), later passes carry it.
// RB = 9 (experiment, BWTC_RADIX9=1; MEASURED SLOWER: one 9-bit pass over the 32 MiB block's records takes 0.272 ms against
// 0.220 ms, so 7 of them lose to 8 eight-bit passes — profiles/r02_experiments.md): nine-bit digits (512 bins; a
// 55..63-bit key then takes 7 passes instead of 8).  The CTA keeps its shape: every
// thread owns digits tid and tid + 256 — two status words per tile row of 512, two look-back walks interleaved in one
// loop (LB_BATCH9 words each in flight) — and the per-warp histograms hold the two digits of a thread as the 16-bit
// halves of one word (a tile has 4096 records, so neither the counts nor the tile-local offsets overflow a half):
// zeroing, the scan over warps and the offset fold cost what they cost with 256 bins.
template <typename KeyT, int BLOCK, int IPT, bool IOTA, bool AUX = false, int RB = 8>
__global__ void __launch_bounds__(BLOCK, (sizeof(KeyT) == 4 && !AUX) ? BWTC_RS_MINB32 : BWTC_RS_MINB) k_radix_pass(const KeyT* __restrict__ keys_in,
                                                      const uint32_t* __restrict__ vals_in,
                                                      KeyT* __restrict__ keys_out, uint32_t* __restrict__ vals_out,
                                                      uint32_t n, uint32_t shift,
                                                      const uint32_t* __restrict__ ghist,
                                                      uint32_t* __restrict__ status, uint32_t* __restrict__ ctrl,
                                                      uint32_t ctr_slot, uint32_t iota_top, uint32_t pack_bits,
                                                      uint32_t topshift, uint32_t pred_mask,
                                                      const uint8_t* __restrict__ aux_in = nullptr,
                                                      uint8_t* __restrict__ aux_out = nullptr) {
  // IOTA: ids are generated (position g holds suffix iota_top - g).  pack_bits != 0 additionally stores, above
  // bit pack_bits of the id, the dense code of the character PRECEDING the suffix — the top character of the
  // next key in the array — so the BWT emission of k_rerank needs no text gather at all.
  static_assert(BLOCK >= 256 && BLOCK % 32 == 0, "BLOCK must cover the 256 digit bins");
  static_assert(RB == 8 || (RB == 9 && BLOCK == 256), "9-bit digits: two digits per thread of a 256-thread CTA");
  constexpr int TILE = BLOCK * IPT, WARPS = BLOCK / 32;
  constexpr uint32_t BINS = 1u << RB, DMASK = BINS - 1u;
  static_assert(TILE <= 65536, "local positions are kept as uint16");
  static_assert(RB == 8 || 2 * TILE < 65536, "9-bit digits: tile-local offsets live in 16-bit halves");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  KeyT* s_keys = reinterpret_cast<KeyT*>(smem_raw);
  uint32_t* s_vals = reinterpret_cast<uint32_t*>(smem_raw + sizeof(KeyT) * TILE);  // ids staged beside the keys
  uint32_t* s_whist = s_vals + TILE;
  uint32_t* s_binbase = s_whist + WARPS * 256;
  uint32_t* s_misc = s_binbase + BINS;  // [0] tile id, [8..23] scan scratch
  uint8_t* s_aux = reinterpret_cast<uint8_t*>(s_misc + 32);  // AUX: bytes staged beside keys and ids

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef BWTC_PROFILE_STAGES
  const unsigned long long t_entry = clock64();
#endif
  // Tile id.  ctr_slot == CTR_STATIC: the block index — CTAs of a 1-D grid are dispatched in index order, so every
  // tile a CTA can wait for (lower ids only) is already resident or finished; measured 4-7% faster than taking a
  // ticket (no atomic + broadcast in front of the loads).  The order is not an architectural guarantee: the spin
  // watchdog turns a violation into an error, and the host then repeats the block with tickets (ctr_slot = a
  // zeroed ctrl word), which are safe under any dispatch order.
  uint32_t tile = blockIdx.x;
  if (ctr_slot == CTR_STATIC_REV) {
    tile = gridDim.x - 1u - blockIdx.x;
  } else if (ctr_slot != CTR_STATIC) {
    if (tid == 0) s_misc[0] = atomicAdd(&ctrl[ctr_slot], 1u);
    __syncthreads();
    tile = s_misc[0];
  }
  // Sticky error word: once a watchdog has fired anywhere in this block's kernel sequence, every later CTA returns
  // before it touches a buffer (the load is issued here, next to the record loads, and tested behind them).
  // (a plain load, not an asm volatile one: it must not fence the record loads below; kernel boundaries make the word
  // visible, and a CTA that misses a concurrent failure merely finishes its tile)
  const uint32_t err_at_entry = ctrl[CTR_ERR];
  // (the per-warp histograms are zeroed AFTER the loads have been issued: their latency covers the zeroing and
  // the barrier)
#ifdef BWTC_PROFILE_STAGES
  if (tid == 0 && g_prof_buf) g_prof_buf[(size_t)tile * 16 + 0] = t_entry;
#endif
  BWTC_PROF(1);
  const uint32_t tile_base = tile * (uint32_t)TILE;
  if (tile_base >= n) return;  // cannot happen with grid == ceil(n / TILE); defensive
  const uint32_t valid = (n - tile_base < (uint32_t)TILE) ? (n - tile_base) : (uint32_t)TILE;

  // ---- load (warp-striped)
  KeyT key[IPT];
  uint32_t val[IPT];
  uint32_t aux[AUX ? IPT / 4 : 1];  // one byte per record, four to a register
#pragma unroll
  for (int q = 0; q < (AUX ? IPT / 4 : 1); ++q) aux[q] = 0;
  const uint32_t first = tile_base + warp * (32 * IPT) + lane;
  if (valid == (uint32_t)TILE) {
#pragma unroll
    for (int k = 0; k < IPT; ++k) key[k] = BWTC_LD(keys_in + first + 32 * k);
#pragma unroll
    for (int k = 0; k < IPT; ++k) val[k] = IOTA ? (iota_top - (first + 32 * k)) : BWTC_LD(vals_in + first + 32 * k);
    if (IOTA && pack_bits) {
#pragma unroll
      for (int k = 0; k < IPT; ++k) {
        const uint32_t g1 = first + 32 * k + 1u;
        const uint32_t pc = (g1 < n) ? ((uint32_t)(keys_in[g1] >> topshift) & pred_mask) : 0u;  // L1 hit: the neighbour's key
        val[k] |= pc << pack_bits;
      }
    }
    if (AUX) {
#pragma unroll
      for (int k = 0; k < IPT; ++k) {
        const uint32_t g = first + 32 * k;
        uint32_t a;
        if (IOTA) a = (g + 1u < n) ? ((uint32_t)(keys_in[g + 1u] >> topshift) & pred_mask) : 0u;
        else a = aux_in[g];
        aux[k / 4] |= a << (8 * (k % 4));
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      const uint32_t g = first + 32 * k;
      key[k] = (g < n) ? keys_in[g] : (KeyT)~(KeyT)0;  // pads: the last digit, last in index order
      val[k] = (g < n) ? (IOTA ? (iota_top - g) : vals_in[g]) : 0u;
      if (IOTA && pack_bits && g + 1u < n) val[k] |= ((uint32_t)(keys_in[g + 1u] >> topshift) & pred_mask) << pack_bits;
      if (AUX) {
        uint32_t a = 0;
        if (IOTA) a = (g + 1u < n) ? ((uint32_t)(keys_in[g + 1u] >> topshift) & pred_mask) : 0u;
        else if (g < n) a = aux_in[g];
        aux[k / 4] |= a << (8 * (k % 4));
      }
    }
  }

  if (err_at_entry) return;
  for (int i = lane; i < 256; i += 32) s_whist[warp * 256 + i] = 0;  // each warp zeroes (and then ranks into) its own
  __syncwarp();
#ifdef BWTC_PROFILE_STAGES
  {
    KeyT acc = 0;
#pragma unroll
    for (int k = 0; k < IPT; ++k) acc ^= key[k] ^ (KeyT)val[k];
    if (acc == (KeyT)0x123456789ABCDEFull) s_misc[1] = 1;  // forces the loads to land before stamp 2
    __syncthreads();
    BWTC_PROF(2);
  }
#endif
  uint32_t cnt = 0, pub = 0;
  uint32_t* my_status = status + (size_t)tile * BINS + (tid & 255);
  // ---- rank inside the warp
  uint16_t lpos[IPT];
  uint32_t* my_hist = s_whist + warp * 256;
  const uint32_t lt = lanemask_lt();
#pragma unroll
  for (int k = 0; k < IPT; ++k) {
    const uint32_t d = (uint32_t)(key[k] >> shift) & DMASK;
    uint32_t m;
    if constexpr (RB == 9) m = match_digit9(d);
    else m = match_digit8(d);
    const int leader = __ffs(m) - 1;
    uint32_t old = 0;
    if constexpr (RB == 9) {
      const uint32_t hs = (d >> 8) * 16u;  // digit d lives in half d >> 8 of word d & 255
      if (lane == leader) old = atomicAdd(&my_hist[d & 255u], (uint32_t)__popc(m) << hs);
      old = (__shfl_sync(0xFFFFFFFFu, old, leader) >> hs) & 0xFFFFu;
    } else {
      if (lane == leader) old = atomicAdd(&my_hist[d], (uint32_t)__popc(m));  // one shared-memory RMW, not LDS+STS
      old = __shfl_sync(0xFFFFFFFFu, old, leader);
    }
    lpos[k] = (uint16_t)(old + __popc(m & lt));
    __syncwarp();
  }
  __syncthreads();
  BWTC_PROF(4);
  if constexpr (RB == 9) {
    // ---- two digits per thread (tid -> low half, tid + 256 -> high half of every packed word)
    uint32_t run = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) {
      const uint32_t t = s_whist[w * 256 + tid];
      s_whist[w * 256 + tid] = run;
      run += t;
    }
    const uint32_t cnt0 = run & 0xFFFFu, cnt1 = run >> 16;
    const uint32_t pub0 = cnt0;
    const uint32_t pub1 = cnt1 - ((tid == 255) ? ((uint32_t)TILE - valid) : 0u);  // pads (digit 511) are not records
    const uint32_t first_flag = (tile == 0 ? LB_PREFIX : 0u);
    st_relaxed_u32(my_status, first_flag | (pub0 + 1u));
    st_relaxed_u32(my_status + 256, first_flag | (pub1 + 1u));
    // tile-local exclusive offsets of both halves with ONE packed scan (every partial sum is <= TILE)
    uint32_t tot_pk = 0, dummy0, dummy1;
    uint32_t pk_excl;
    scan256_excl2(run, 0u, s_misc + 8, pk_excl, dummy0, tot_pk, dummy1);
    const uint32_t texcl0 = pk_excl & 0xFFFFu;
    const uint32_t texcl1 = (pk_excl >> 16) + (tot_pk & 0xFFFFu);
    uint32_t gexcl0, gexcl1, gtot0, gtot1;
    scan256_excl2(ghist[tid], ghist[tid + 256], s_misc + 8, gexcl0, gexcl1, gtot0, gtot1);
    gexcl1 += gtot0;
    {
      const uint32_t fold = texcl0 | (texcl1 << 16);
#pragma unroll
      for (int w = 0; w < WARPS; ++w) s_whist[w * 256 + tid] += fold;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      const uint32_t d = (uint32_t)(key[k] >> shift) & DMASK;
      const uint32_t p = ((my_hist[d & 255u] >> ((d >> 8) * 16u)) & 0xFFFFu) + lpos[k];
      s_keys[p] = key[k];
      s_vals[p] = val[k];
      if (AUX) s_aux[p] = (uint8_t)(aux[k / 4] >> (8 * (k % 4)));
    }
    BWTC_PROF(5);
    // ---- decoupled look-back of both digits, interleaved: LB_BATCH9 words of each in flight per round trip
    uint32_t excl0 = 0, excl1 = 0;
    if (tile != 0) {
      long long t0 = (long long)tile - 1, t1 = t0;
      uint32_t spins = 0;
      uint32_t live0 = 0xFFFFFFFFu, live1 = 0xFFFFFFFFu;  // all-ones while the digit's walk is not finished
      while (live0 | live1) {
        uint32_t v0[LB_BATCH9], v1[LB_BATCH9];
        const uint32_t* row0 = status + t0 * (long long)BINS + tid;
        const uint32_t* row1 = status + t1 * (long long)BINS + 256 + tid;
#pragma unroll
        for (int i = 0; i < LB_BATCH9; ++i) v0[i] = ld_relaxed_u32(row0 - i * (int)BINS);
#pragma unroll
        for (int i = 0; i < LB_BATCH9; ++i) v1[i] = ld_relaxed_u32(row1 - i * (int)BINS);
        uint32_t alive0 = live0, alive1 = live1, fin0 = 0, fin1 = 0;
        int c0 = 0, c1 = 0;
#pragma unroll
        for (int i = 0; i < LB_BATCH9; ++i) {
          {
            const uint32_t pubd = (uint32_t)((int32_t)(v0[i] | (0u - v0[i])) >> 31);
            const uint32_t ispre = (uint32_t)((int32_t)v0[i] >> 31);
            const uint32_t isagg = pubd & ~ispre;
            excl0 += ((v0[i] & LB_VALUE) - 1u) & alive0 & pubd;
            fin0 |= alive0 & ispre;
            c0 += (int)(alive0 & isagg & 1u);
            alive0 &= isagg;
          }
          {
            const uint32_t pubd = (uint32_t)((int32_t)(v1[i] | (0u - v1[i])) >> 31);
            const uint32_t ispre = (uint32_t)((int32_t)v1[i] >> 31);
            const uint32_t isagg = pubd & ~ispre;
            excl1 += ((v1[i] & LB_VALUE) - 1u) & alive1 & pubd;
            fin1 |= alive1 & ispre;
            c1 += (int)(alive1 & isagg & 1u);
            alive1 &= isagg;
          }
        }
        live0 &= ~fin0;  // fin is all-ones once the walk met an inclusive prefix
        live1 &= ~fin1;
        t0 -= c0;
        t1 -= c1;
        if ((live0 | live1) && c0 + c1 == 0) {
          ++spins;
          if (spins > g_lb_spin_limit || ((spins & 255u) == 0u && ld_relaxed_u32(ctrl + CTR_ERR))) {
            atomicExch(&ctrl[CTR_ERR], 1u);
            break;
          }
          __nanosleep(20);
        }
      }
      st_relaxed_u32(my_status, LB_PREFIX | ((excl0 + pub0 + 1u) & LB_VALUE));
      st_relaxed_u32(my_status + 256, LB_PREFIX | ((excl1 + pub1 + 1u) & LB_VALUE));
    }
    s_binbase[tid] = gexcl0 + excl0 - texcl0;
    s_binbase[tid + 256] = gexcl1 + excl1 - texcl1;
    __syncthreads();
    BWTC_PROF(6);
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      const uint32_t p = tid + k * BLOCK;
      const KeyT kk = s_keys[p];
      const uint32_t vv = s_vals[p];
      const uint32_t d = (uint32_t)(kk >> shift) & DMASK;
      const uint32_t g = s_binbase[d] + p;
      if (p < valid) {
        BWTC_ST(keys_out + g, kk);
        BWTC_ST(vals_out + g, vv);
        if (AUX) aux_out[g] = s_aux[p];
      }
    }
    BWTC_PROF(8);
    return;
  }

  // ---- per-digit: exclusive scan over warps; tile-local and global exclusive digit offsets
  if (tid < 256) {
    uint32_t run = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) {
      const uint32_t t = s_whist[w * 256 + tid];
      s_whist[w * 256 + tid] = run;
      run += t;
    }
    cnt = run;
    pub = cnt;
    if (tid == 255) pub -= ((uint32_t)TILE - valid);  // pads are not records
    st_relaxed_u32(my_status, (tile == 0 ? LB_PREFIX : 0u) | (pub + 1u));
  }
  const uint32_t texcl = scan256_excl(cnt, s_misc + 8);
  const uint32_t gcount = (tid < 256) ? ghist[tid] : 0u;
  const uint32_t gexcl = scan256_excl(gcount, s_misc + 8);
  if (tid < 256) {
    // fold the tile-local digit offset into every warp's offset: staging then needs ONE digit-indexed lookup
#pragma unroll
    for (int w = 0; w < WARPS; ++w) s_whist[w * 256 + tid] += texcl;
  }
  __syncthreads();

  // ---- ... stage keys in sorted order (needs tile-local offsets only) while predecessors publish
#pragma unroll
  for (int k = 0; k < IPT; ++k) {
    const uint32_t d = (uint32_t)(key[k] >> shift) & 0xFFu;
    const uint32_t p = my_hist[d] + lpos[k];
    s_keys[p] = key[k];
    s_vals[p] = val[k];
    if (AUX) s_aux[p] = (uint8_t)(aux[k / 4] >> (8 * (k % 4)));
  }

  BWTC_PROF(5);
  // ---- decoupled look-back, one digit per thread, LB_BATCH predecessor words in flight per round trip
  if (tid < 256) {
    uint32_t excl = 0;
    if (tile != 0) {
      long long t = (long long)tile - 1;
      uint32_t spins = 0;
      bool done = false;
#ifdef BWTC_PROFILE_STAGES
      uint32_t prof_iters = 0;
#endif
      while (!done) {
#ifdef BWTC_PROFILE_STAGES
        ++prof_iters;
#endif
        uint32_t v[LB_BATCH];
        const uint32_t* row = status + (long long)t * 256 + tid;  // rows t, t-1, ...; rows -1..-LB_PAD_ROWS are "prefix 0"
#pragma unroll
        for (int i = 0; i < LB_BATCH; ++i) v[i] = ld_relaxed_u32(row - i * 256);
        // branch-free walk: `alive` is all-ones while every word so far was an aggregate
        uint32_t alive = 0xFFFFFFFFu, fin = 0;
        int consumed = 0;
#pragma unroll
        for (int i = 0; i < LB_BATCH; ++i) {
          const uint32_t pubd = (uint32_t)((int32_t)(v[i] | (0u - v[i])) >> 31);  // published (non-zero) -> ~0
          const uint32_t ispre = (uint32_t)((int32_t)v[i] >> 31);                 // bit 31 -> 0 / ~0
          const uint32_t isagg = pubd & ~ispre;
          excl += ((v[i] & LB_VALUE) - 1u) & alive & pubd;
          fin |= alive & ispre;
          consumed += (int)(alive & isagg & 1u);
          alive &= isagg;
        }
        done = fin != 0;
        t -= consumed;
        if (!done && consumed == 0) {
          ++spins;
          if (spins > g_lb_spin_limit || ((spins & 255u) == 0u && ld_relaxed_u32(ctrl + CTR_ERR))) {
            atomicExch(&ctrl[CTR_ERR], 1u);  // (or somebody else's watchdog fired: stop waiting for a tile that gave up)
            break;
          }
          __nanosleep(20);
        }
      }
      st_relaxed_u32(my_status, LB_PREFIX | ((excl + pub + 1u) & LB_VALUE));
#ifdef BWTC_PROFILE_STAGES
      if (tid == 0 && g_prof_buf) {
        g_prof_buf[(size_t)tile * 16 + 9] = prof_iters;
        g_prof_buf[(size_t)tile * 16 + 10] = spins;
        g_prof_buf[(size_t)tile * 16 + 11] = clock64();
        g_prof_buf[(size_t)tile * 16 + 12] = (unsigned long long)((long long)tile - 1 - t);
      }
#endif
    }
    s_binbase[tid] = gexcl + excl - texcl;  // + local position = global position (mod 2^32)
  }
  __syncthreads();
  BWTC_PROF(6);
  // one scatter loop writes key and id of a record (both staged in sorted order).  (An unpredicated full-tile
  // variant of this loop was measured 5% SLOWER: the compiler then issues all 32 stores as one burst.)
#pragma unroll
  for (int k = 0; k < IPT; ++k) {
    const uint32_t p = tid + k * BLOCK;
    const KeyT kk = s_keys[p];
    const uint32_t vv = s_vals[p];
    const uint32_t d = (uint32_t)(kk >> shift) & 0xFFu;
    const uint32_t g = s_binbase[d] + p;
    if (p < valid) {
      BWTC_ST(keys_out + g, kk);
      BWTC_ST(vals_out + g, vv);
      if (AUX) aux_out[g] = s_aux[p];
    }
  }
  BWTC_PROF(8);
}

// =====================================================================================================
// k_rerank — segmented re-ranking after a sort round.  Over the sorted records j = 0..m-1:
//   headfull(j): the full key differs from its predecessor's (ROUND0: or the predecessor's window ran past
//                the end of the text — such a suffix is unique and precedes its equal-key neighbours);
//   headhi(j)  : the old group (high key part) changes (ROUND0: only j = 0).
//   HF(j), HH(j) = position of the last headfull / headhi at or before j  (two max-scans: thread-local,
//                  warp shuffles, CTA, and a single 64-bit decoupled look-back word across tiles);
//   new rank   = old_rank + HF(j) - HH(j)   (ROUND0: HF(j));   singleton = headfull(j) && headfull(j+1).
// rank[idx[j]] is scattered only when it changes or becomes final (directly, per id window, or staged per id
// bucket for k_scatter_bucket).  Records left in non-singleton groups are staged in sorted order per tile
// (StageParams) and counted in ctrl[CTR_LIVE]; the largest group goes to ctrl[CTR_MAXGROUP].
// Replaces the rank assignment of sort_typeBstar (divsufsort.c:147-158) and tr_partition / tr_copy
// bookkeeping (trsort.c:220-323), negative-run skipping (trsort.c:563-585).
// =====================================================================================================
struct RerankParams {
  uint32_t m;             // records
  uint32_t short_thresh;  // ROUND0: suffix ids >= this have a window running past the text end
  int lo_bits;            // width of the low key part (rounds >= 1)
  uint32_t win_lo, win_hi;  // only suffix ids in [win_lo, win_hi) are written / counted by this launch: the rank
                            // scatter of a big block is split into windows that stay L2-resident (random 4-byte
                            // writes into a >L2 array cost a DRAM sector fill + write-back each)
  uint32_t ctr_slot;        // CTR_STATIC (tile id = block index) or the ctrl word used as tile ticket counter
  uint32_t id_mask;         // ROUND0: the sorted payload is id | code(T[id-1]) << id_bits when packed != 0
  uint32_t id_bits;
  uint32_t packed;          // 1: predecessor code above the id; 2: predecessor codes in pred_aux[] (sorted order)
  const uint8_t* pred_aux;
  uint8_t decode[256];      // dense code -> byte (packed emission)
  uint32_t nbuckets;        // > 1: bucketed scatter — instead of writing rank[] the tile stages its (id, rank) pairs
  uint32_t bucket_magic;    //      grouped by id bucket (bucket = min(umulhi(id, magic), nbuckets-1)); see k_scatter_bucket
  uint32_t* nr_out;         // != nullptr: additionally store every record's new rank word at its SORTED position (0xFFFFFFFF =
                            // "rank unchanged"), coalesced; k_scatter_window then serves the other id windows from
                            // (idx[], nr_out[]) without repeating the re-rank
  uint32_t direct0;         // bucketed: ids of bucket 0 are written to rank[] directly (its window stays L2-resident during
                            // this launch), only the other buckets are staged — the two-window case: one pass over the
                            // records + one k_scatter_bucket over half of the pairs, instead of two passes over the records
  // ROUND0, lazy ranks (DESIGN.md §3.9): 1 = rank[] is written only for suffixes that stay in a group (and the few "short"
  // ones), their bit is set in livebits, and the first sorted position of every key prefix goes to ktab; a singleton's
  // rank is its sorted position and is looked up in the retained sorted keys when somebody needs it (rank_lookup).
  // 2 = materialise: write rank[] for the singletons only (the fallback out of lazy mode; nothing else is touched).
  uint32_t lazy;
  // Which records this launch emits BWT bytes for — 0: those whose id is in [win_lo, win_hi); 1: all (round 0: the first
  // launch of a windowed scatter, so a thread's eight consecutive output bytes leave as one store; any round: the only
  // k_rerank launch when k_scatter_window serves the other window); 2: none.
  uint32_t emit;
  // > 0: every CTA first asks L2 for the records of tile (mine + pf_tiles) — the tile a CTA launched about one wave later
  // will load; the kernel is bound by the latency of its up-front record loads (ncu: 49% of stall samples on their first use)
  uint32_t pf_tiles;
  uint32_t* livebits;
  uint32_t* ktab;
  uint32_t tshift;          // key >> tshift = table index
};

// What a consumer of ranks needs in lazy mode (by value in the kernel arguments).
struct LookupParams {
  uint32_t enabled;          // 0: rank[] is complete, plain loads
  uint32_t keybytes;         // 4 or 8: type of the sorted round-0 keys
  const void* sorted_keys;   // N keys in sorted order
  const uint32_t* ktab;      // (1 << tbits) + 1 entries: first sorted position whose key prefix is >= the index
  const uint32_t* livebits;  // bit i set: rank[i] is valid
  const uint8_t* text;
  uint32_t N, bits, chars, tshift;
  uint32_t rbits;            // PackParams::rbits of the round-0 keys
  uint8_t lut[256];
};

// Lower bound of `key` in sorted[lo, hi) reading whole 32-byte sectors: the first probe is INTERPOLATED from the key bits
// below the table prefix (inside one table bucket they are close to uniform), then the search walks to the neighbouring
// sector twice before it falls back to bisection.  A bucket of ~32 keys costs 1-2 DRAM sectors instead of the ~3 distinct
// ones of a plain binary search.  The key array is padded to a sector.  Only the tail of a lazy block searches (k_small_rounds:
// <= 2048 look-ups per round in one CTA, k_finish: <= 257), so what counts is the chain of dependent DRAM round trips.
template <typename KeyT>
__device__ __forceinline__ uint32_t sector_lower_bound(const KeyT* __restrict__ sk, KeyT key, uint32_t lo, uint32_t hi,
                                                       uint32_t frac16) {
  constexpr uint32_t KPS = 32 / sizeof(KeyT);  // keys per sector
  uint32_t g = lo + (uint32_t)(((unsigned long long)(hi - lo) * frac16) >> 16);
  for (int it = 0; lo < hi; ++it) {
    if (g >= hi) g = hi - 1u;
    if (g < lo) g = lo;
    const uint32_t s = g & ~(KPS - 1u);
    KeyT v[KPS];
    if constexpr (sizeof(KeyT) == 8) {
      const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(sk + s);
      const ulonglong2 y = *reinterpret_cast<const ulonglong2*>(sk + s + 2);
      v[0] = (KeyT)x.x; v[1] = (KeyT)x.y; v[2] = (KeyT)y.x; v[3] = (KeyT)y.y;
    } else {
      const uint4 x = *reinterpret_cast<const uint4*>(sk + s);
      const uint4 y = *reinterpret_cast<const uint4*>(sk + s + 4);
      v[0] = (KeyT)x.x; v[1] = (KeyT)x.y; v[2] = (KeyT)x.z; v[3] = (KeyT)x.w;
      v[4] = (KeyT)y.x; v[5] = (KeyT)y.y; v[6] = (KeyT)y.z; v[7] = (KeyT)y.w;
    }
    const uint32_t a = s > lo ? s : lo, b = (s + KPS < hi) ? s + KPS : hi;  // valid entries of this sector
    uint32_t c = 0;
#pragma unroll
    for (uint32_t q = 0; q < KPS; ++q) c += (s + q >= a && s + q < b && v[q] < key) ? 1u : 0u;
    if (c == 0u) {            // nothing below the key here: the bound is at or left of a
      hi = a;
      g = (it < 2) ? (a ? a - 1u : 0u) : lo + ((hi - lo) >> 1);
    } else if (c == b - a) {  // everything here is below the key: the bound is at or right of b
      lo = b;
      g = (it < 2) ? b : lo + ((hi - lo) >> 1);
    } else {
      return a + c;
    }
  }
  return lo;
}

// The round-0 key of suffix j, as k_pack_round0 builds it (windows past the end of the text padded with code 0).
__device__ __forceinline__ unsigned long long round0_key(const LookupParams& lk, uint32_t j) {
  unsigned long long key = 0;
  for (uint32_t c = 0; c < lk.chars; ++c) {
    const uint32_t g = j + c;
    key = (key << lk.bits) | (unsigned long long)((g < lk.N) ? lk.lut[lk.text[g]] : 0u);
  }
  if (lk.rbits) {
    const uint32_t g = j + lk.chars;
    key = (key << lk.rbits) | (unsigned long long)(((g < lk.N) ? (uint32_t)lk.lut[lk.text[g]] : 0u) >> (lk.bits - lk.rbits));
  }
  return key;
}

// rank of suffix j (without the DONE flag).
__device__ __forceinline__ uint32_t rank_lookup(const LookupParams& lk, const uint32_t* __restrict__ rank, uint32_t j) {
  if (!lk.enabled || ((lk.livebits[j >> 5] >> (j & 31u)) & 1u)) return rank[j] & RANK_MASK;
  const unsigned long long key = round0_key(lk, j);
  const uint32_t p = (uint32_t)(key >> lk.tshift);
  uint32_t lo = lk.ktab[p], hi = lk.ktab[p + 1u];
  // the 16 key bits below the table prefix, as a fraction of the bucket
  const uint32_t frac16 = lk.tshift >= 16u ? (uint32_t)(key >> (lk.tshift - 16u)) & 0xFFFFu
                                           : ((uint32_t)key << (16u - lk.tshift)) & 0xFFFFu;
  if (lk.keybytes == 8u)
    return sector_lower_bound<unsigned long long>(static_cast<const unsigned long long*>(lk.sorted_keys), key, lo, hi, frac16);
  return sector_lower_bound<uint32_t>(static_cast<const uint32_t*>(lk.sorted_keys), (uint32_t)key, lo, hi, frac16);
}

// ktab holds the first sorted position of every key prefix that occurs (k_rerank, lazy) and 0xFFFFFFFF elsewhere; fill the
// holes from the right (suffix minimum) so that [ktab[p], ktab[p+1]) is the position range of prefix p.  ktab[entries] = N.
// Two small kernels over chunks of KTAB_CHUNK entries: chunk minima, then every chunk takes the minimum of the chunks to
// its right as its carry and fills itself.  (A single-CTA sweep over the 2^20 entries took 0.6 ms.)
constexpr uint32_t KTAB_CHUNK = 4096;  // 256 threads x 16

__global__ void __launch_bounds__(256) k_ktab_chunkmin(const uint32_t* __restrict__ ktab, uint32_t entries, uint32_t* __restrict__ cmin) {
  __shared__ uint32_t s_w[8];
  const uint32_t base = blockIdx.x * KTAB_CHUNK + threadIdx.x * 16u;
  uint32_t mn = 0xFFFFFFFFu;
#pragma unroll
  for (int k = 0; k < 16; ++k)
    if (base + k < entries) mn = min(mn, ktab[base + k]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(0xFFFFFFFFu, mn, o));
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = mn;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0xFFFFFFFFu;
    for (int w = 0; w < 8; ++w) t = min(t, s_w[w]);
    cmin[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(256) k_ktab_fill(uint32_t* __restrict__ ktab, uint32_t entries, uint32_t N,
                                                   const uint32_t* __restrict__ cmin, uint32_t nchunks) {
  __shared__ uint32_t s_w[8];
  __shared__ uint32_t s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // carry = first position of any prefix in the chunks to the right (N if none)
  uint32_t c = N;
  for (uint32_t q = blockIdx.x + 1u + tid; q < nchunks; q += 256) c = min(c, cmin[q]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c = min(c, __shfl_xor_sync(0xFFFFFFFFu, c, o));
  if (lane == 0) s_w[warp] = c;
  __syncthreads();
  if (tid == 0) {
    uint32_t t = N;
    for (int w = 0; w < 8; ++w) t = min(t, s_w[w]);
    s_carry = t;
    if (blockIdx.x == nchunks - 1u) ktab[entries] = N;
  }
  __syncthreads();
  const uint32_t carry = s_carry;
  // thread tid owns 16 entries; thread 255 the highest.  Suffix minimum: from the right.
  const uint32_t base = blockIdx.x * KTAB_CHUNK + (uint32_t)tid * 16u;
  uint32_t v[16];
  uint32_t mn = 0xFFFFFFFFu;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    v[k] = (base + k < entries) ? ktab[base + k] : 0xFFFFFFFFu;
    mn = min(mn, v[k]);
  }
  // exclusive suffix-min over threads: min of the threads to my right
  uint32_t inc = mn;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_down_sync(0xFFFFFFFFu, inc, o);
    if (lane + o < 32) inc = min(inc, t);
  }
  __syncthreads();
  if (lane == 0) s_w[warp] = inc;
  uint32_t ex = __shfl_down_sync(0xFFFFFFFFu, inc, 1);
  if (lane == 31) ex = 0xFFFFFFFFu;
  __syncthreads();
  for (int w = warp + 1; w < 8; ++w) ex = min(ex, s_w[w]);
  uint32_t run = min(ex, carry);
#pragma unroll
  for (int k = 15; k >= 0; --k) {
    run = min(run, v[k]);
    if (base + k < entries) ktab[base + k] = run;
  }
}

// Live-record staging of k_rerank.  The window launch with sp.enable != 0 writes, for EVERY record of its tile
// that stays in a non-singleton group (whatever its id window), the pair (new rank, id) in sorted order to
// stage_*[tile_base + 0 .. cnt) and the count to tile_cnt[tile]; it also owns ctrl[CTR_LIVE] / [CTR_MAXGROUP].
// k_scan_tile_counts + k_gather_chunks later concatenate the chunks — in tile order, so every group stays
// contiguous — into the compact lists that k_seg_round, k_small_rounds and k_build_from_list consume.
struct StageParams {
  uint32_t* stage_nr;
  uint32_t* stage_id;
  uint32_t* tile_cnt;
  int enable;
  // bucketed rank scatter (RerankParams::nbuckets > 1): records of tile t, grouped by id bucket, go to
  // sc_*[tile_base + tile_woff[t*(nbuckets+1) + b] ..); k_scatter_bucket then writes one bucket (= one L2-resident
  // window of rank[]) per launch, reading every staged record exactly once.
  uint32_t* sc_id;
  uint32_t* sc_nr;
  uint32_t* tile_woff;
};

// BWT emission fused into the re-rank: the moment a suffix becomes a singleton its rank is final, the records
// are at hand in SORTED order, so L[rank] = T[id-1] is written with (nearly) consecutive addresses and only the
// text gather (L2-resident) is random.  No separate N-element byte scatter remains.  The one byte that the block
// contract moves into the hole (L[N-1] -> out[pidx]) is parked in *lastch for k_finish.
struct EmitParams {
  const uint8_t* text;
  uint8_t* out;
  uint32_t* lastch;  // bit 8 set = valid; one word per block of a batch
  uint32_t N;
  int block_mode;
  // Batch of nblocks > 1 small blocks sorted as ONE text (DESIGN.md §3.6): block k owns the suffix ids AND the
  // ranks [k*stride, k*stride + N_k) — the block number is the most significant part of every sort key.
  uint32_t nblocks;
  uint32_t stride;
  // Suffix array of a raw text (bwtc_cuda_divsufsort, DESIGN.md §3.11): sa[rank] = id for EVERY singleton, suffix 0
  // included.  Only the SA = true instantiations of k_rerank / k_seg_round / k_small_rounds read it (null otherwise), so
  // the kernels of every other call are the ones they were without it.
  int32_t* sa;
};

// Suffix 0 of a block owns the hole at pidx: it has no preceding character to emit.
__device__ __forceinline__ bool owns_hole(const EmitParams& ep, uint32_t id) {
  return ep.nblocks <= 1u ? (id == 0u) : (id % ep.stride == 0u);
}

// L[nr] = ch.  The one byte the block contract moves into the hole (L[N-1] -> out[pidx]) is parked for k_finish.
__device__ __forceinline__ void emit_bwt(const EmitParams& ep, uint32_t nr, uint8_t ch) {
  if (ep.nblocks <= 1u) {
    if (ep.block_mode && nr == ep.N - 1u) *ep.lastch = 0x100u | ch;
    else ep.out[nr] = ch;
    return;
  }
  const uint32_t k = nr / ep.stride;
  const uint32_t last = ((k + 1u == ep.nblocks) ? ep.N : (k + 1u) * ep.stride) - 1u;
  if (nr == last) ep.lastch[k] = 0x100u | ch;
  else ep.out[nr] = ch;
}

template <typename KeyT, bool ROUND0, bool LAZY = false, bool SA = false>
__global__ void __launch_bounds__(256, (ROUND0 && !LAZY) ? 5 : 4) k_rerank(const KeyT* __restrict__ keys, const uint32_t* __restrict__ idx,
                                                uint32_t* __restrict__ rank, RerankParams rp,
                                                unsigned long long* __restrict__ tstate,
                                                uint32_t* __restrict__ ctrl, EmitParams ep, StageParams sp) {
  constexpr int BLOCK = 256, IPT = 8, TILE = BLOCK * IPT, WARPS = BLOCK / 32;
  __shared__ KeyT s_lastkey[BLOCK];
  __shared__ uint32_t s_lastshort[BLOCK];
  __shared__ uint32_t s_firsthead[BLOCK + 1];
  __shared__ uint32_t s_wf[WARPS], s_wh[WARPS];
  __shared__ uint32_t s_tile, s_cf, s_ch, s_firsth0;
  __shared__ uint32_t s_bcnt[MAX_RERANK_WINDOWS + 1];
  __shared__ uint8_t s_dec[ROUND0 ? 256 : 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // tile id: the block index, or a ticket in the watchdog-fallback mode (see k_radix_pass).  s_bcnt / s_dec are first
  // read behind later barriers, so the block-index path needs no barrier in front of the loads.
  uint32_t tile = blockIdx.x;
  if (ROUND0 && rp.packed) s_dec[tid] = rp.decode[tid];
  if (tid <= MAX_RERANK_WINDOWS) s_bcnt[tid] = 0;
  if (rp.ctr_slot == CTR_STATIC_REV) {
    tile = gridDim.x - 1u - blockIdx.x;
  } else if (rp.ctr_slot != CTR_STATIC) {
    if (tid == 0) s_tile = atomicAdd(&ctrl[rp.ctr_slot], 1u);
    __syncthreads();
    tile = s_tile;
  }
  const uint32_t err_at_entry = ctrl[CTR_ERR];  // sticky: an earlier kernel of this block failed (see k_radix_pass);
                                                // a plain load, tested behind the record loads it is issued with
  const uint32_t m = rp.m;
  const uint32_t tile_base = tile * (uint32_t)TILE;
  if (tile_base >= m) return;
  const uint32_t j0 = tile_base + tid * IPT;
  KeyT key[IPT];
  uint32_t id[IPT];
  if (tile_base + TILE <= m) {  // full tile: 128-bit loads (buffers are 256-byte aligned, j0 % 8 == 0)
    if (sizeof(KeyT) == 8) {
      const ulonglong2* pk = reinterpret_cast<const ulonglong2*>(keys + j0);
#pragma unroll
      for (int q = 0; q < IPT / 2; ++q) {
        const ulonglong2 v = __ldcs(pk + q);
        key[2 * q] = (KeyT)v.x;
        key[2 * q + 1] = (KeyT)v.y;
      }
    } else {
      const uint4* pk = reinterpret_cast<const uint4*>(keys + j0);
#pragma unroll
      for (int q = 0; q < IPT / 4; ++q) {
        const uint4 v = __ldcs(pk + q);
        key[4 * q] = (KeyT)v.x; key[4 * q + 1] = (KeyT)v.y; key[4 * q + 2] = (KeyT)v.z; key[4 * q + 3] = (KeyT)v.w;
      }
    }
    const uint4* pi = reinterpret_cast<const uint4*>(idx + j0);
#pragma unroll
    for (int q = 0; q < IPT / 4; ++q) {
      const uint4 v = __ldcs(pi + q);
      id[4 * q] = v.x; id[4 * q + 1] = v.y; id[4 * q + 2] = v.z; id[4 * q + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      const uint32_t j = j0 + k;
      key[k] = (j < m) ? keys[j] : (KeyT)0;
      id[k] = (j < m) ? idx[j] : 0u;
    }
  }
  if (err_at_entry) return;
  // (issued once my own record loads have landed: the DRAM queue is idle while the resident CTAs scan)
  if (rp.pf_tiles) {
    const unsigned long long pbase = ((unsigned long long)tile + rp.pf_tiles) * (unsigned long long)TILE;
    if (pbase + TILE <= (unsigned long long)m) {
      constexpr int KLINES = TILE * (int)sizeof(KeyT) / 128, ILINES = TILE * 4 / 128;  // 128 / 64 (u64) or 64 / 64 lines
      const char* p = nullptr;
      if (tid < KLINES) p = reinterpret_cast<const char*>(keys + pbase) + (size_t)tid * 128;
      else if (tid < KLINES + ILINES) p = reinterpret_cast<const char*>(idx + pbase) + (size_t)(tid - KLINES) * 128;
      else if (ROUND0 && rp.packed == 2u && tid < KLINES + ILINES + TILE / 128) p = reinterpret_cast<const char*>(rp.pred_aux + pbase) + (size_t)(tid - KLINES - ILINES) * 128;
      // the address is made to depend on my last loaded record (an opaque "and 0"), so the prefetch issues behind the loads
      uint32_t zero;
      asm volatile("and.b32 %0, %1, 0;" : "=r"(zero) : "r"((uint32_t)key[IPT - 1] ^ id[IPT - 1]));
      if (p) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + zero));
    }
  }

  uint32_t pc0 = 0, pc1 = 0;  // packed predecessor codes of the 8 records (one byte each)
  if (ROUND0 && rp.packed == 2u) {
    if (tile_base + TILE <= m) {
      const uint2 v = *reinterpret_cast<const uint2*>(rp.pred_aux + j0);  // j0 % 8 == 0, buffer 256-byte aligned
      pc0 = v.x;
      pc1 = v.y;
    } else {
#pragma unroll
      for (int k = 0; k < IPT; ++k) {
        const uint32_t c = (j0 + k < m) ? rp.pred_aux[j0 + k] : 0u;
        if (k < 4) pc0 |= c << (8 * k);
        else pc1 |= c << (8 * (k - 4));
      }
    }
  } else if (ROUND0 && rp.packed) {
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      const uint32_t c = id[k] >> rp.id_bits;
      if (k < 4) pc0 |= c << (8 * k);
      else pc1 |= c << (8 * (k - 4));
      id[k] &= rp.id_mask;
    }
  }
  uint32_t lowbits = 0;  // rounds >= 1: bit 0 of each record's old rank travels in bit 31 of the id (k_build_keys)
  if (!ROUND0) {
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      lowbits |= (id[k] >> 31) << k;
      id[k] &= 0x7FFFFFFFu;
    }
  }
  // hand the last key (and its "short" flag) of every thread to its right neighbour
  s_lastkey[tid] = key[IPT - 1];
  if (ROUND0) s_lastshort[tid] = (j0 + IPT - 1 < m && id[IPT - 1] >= rp.short_thresh) ? 1u : 0u;
  __syncthreads();
  KeyT prevkey;
  uint32_t prevshort = 0;
  bool has_prev = true;
  if (tid > 0) {
    prevkey = s_lastkey[tid - 1];
    if (ROUND0) prevshort = s_lastshort[tid - 1];
  } else if (tile_base > 0) {
    prevkey = keys[tile_base - 1];
    if (ROUND0) prevshort = ((idx[tile_base - 1] & rp.id_mask) >= rp.short_thresh) ? 1u : 0u;
  } else {
    prevkey = 0;
    has_prev = false;
  }

  // thread-local flags and running maxima (positions stored +1, 0 = none)
  uint32_t headfull = 0, headhi = 0;  // bit k
  uint32_t lf[IPT], lh[IPT];
  uint32_t runf = 0, runh = 0;
#pragma unroll
  for (int k = 0; k < IPT; ++k) {
    const uint32_t j = j0 + k;
    bool hf, hh;
    if (j >= m) {
      hf = hh = true;  // terminator for singleton detection; never written
    } else if (k == 0 && !has_prev) {
      hf = hh = true;
    } else {
      const KeyT pk = (k == 0) ? prevkey : key[k - 1];
      const uint32_t ps = ROUND0 ? ((k == 0) ? prevshort : ((id[k - 1] >= rp.short_thresh) ? 1u : 0u)) : 0u;
      hf = (key[k] != pk) || (ps != 0);
      hh = ROUND0 ? false : ((key[k] >> rp.lo_bits) != (pk >> rp.lo_bits));
    }
    if (hf) { headfull |= 1u << k; runf = j + 1; }
    if (hh) { headhi |= 1u << k; runh = j + 1; }
    lf[k] = runf;
    lh[k] = runh;
  }
  s_firsthead[tid] = headfull & 1u;
  if (tid == 0) s_firsth0 = headhi & 1u;
  // CTA-wide exclusive max-scan of (runf, runh)
  uint32_t incf = runf, inch = runh;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t tf = __shfl_up_sync(0xFFFFFFFFu, incf, o);
    const uint32_t th = __shfl_up_sync(0xFFFFFFFFu, inch, o);
    if (lane >= o) { incf = max(incf, tf); inch = max(inch, th); }
  }
  if (lane == 31) { s_wf[warp] = incf; s_wh[warp] = inch; }
  uint32_t exf = __shfl_up_sync(0xFFFFFFFFu, incf, 1);
  uint32_t exh = __shfl_up_sync(0xFFFFFFFFu, inch, 1);
  if (lane == 0) { exf = 0; exh = 0; }
  __syncthreads();
  uint32_t aggf = 0, aggh = 0;
#pragma unroll
  for (int w = 0; w < WARPS; ++w) {
    const uint32_t tf = s_wf[w], th = s_wh[w];
    if (w < warp) { exf = max(exf, tf); exh = max(exh, th); }
    aggf = max(aggf, tf);
    aggh = max(aggh, th);
  }
  // Tile look-back.  One 64-bit word per tile, two independent 32-bit components, [63:32] for HH and [31:0] for HF:
  //   0 = not published yet, 0xFFFFFFFF = "no head in this tile" (the carry is still being looked up), anything else =
  //   the final inclusive value (position of the last head + 1, at most 2^31 - 1)
  // A max-scan of positions has a property a sum-scan lacks: a tile that CONTAINS a head already knows its
  // inclusive prefix (its own last head), so it publishes "final" at once and never waits for anybody.  Only
  // a tile whose first record is not a head needs the carry — normally found in the tile right before it —
  // and only a tile with no head at all (inside a group longer than a tile) forwards what it found.
  if (warp == 0) {
    const bool first_is_f = (s_firsthead[0] != 0);          // thread 0's first record is a full-key head
    const bool first_is_h = ROUND0 ? true : (s_firsth0 != 0);
    constexpr uint32_t NOHEAD = 0xFFFFFFFFu;
    constexpr unsigned long long BEFORE_TILE0 = (1ull << 32) | 1ull;  // (never selected: tile 0 always holds a head)
    const uint32_t pubf = aggf, pubh = ROUND0 ? 1u : aggh;
    const uint32_t flagf = pubf ? 2u : 1u, flagh = pubh ? 2u : 1u;
    uint32_t cf = 0, ch = 0;
    if (lane == 0)
      st_relaxed_u64(tstate + tile, ((unsigned long long)(pubh ? pubh : NOHEAD) << 32) | (unsigned long long)(pubf ? pubf : NOHEAD));
    bool needf = !first_is_f && tile > 0, needh = !first_is_h && tile > 0;
    if (needf || needh) {
      long long base = (long long)tile - 1;
      uint32_t spins = 0;
      while (needf || needh) {
        const long long t = base - lane;
        unsigned long long v = (t >= 0) ? ld_relaxed_u64(tstate + t) : BEFORE_TILE0;
        while (v == 0ull) {                                                     // not published yet
          ++spins;
          if (spins > g_lb_spin_limit || ((spins & 255u) == 0u && ld_relaxed_u32(ctrl + CTR_ERR))) {
            atomicExch(&ctrl[CTR_ERR], 2u);
            v = BEFORE_TILE0;
            break;
          }
          __nanosleep(20);
          v = ld_relaxed_u64(tstate + t);
        }
        if (needf) {
          const uint32_t fin = __ballot_sync(0xFFFFFFFFu, (uint32_t)v != NOHEAD);
          if (fin) {
            cf = __shfl_sync(0xFFFFFFFFu, (uint32_t)v, __ffs(fin) - 1);
            needf = false;
          }
        }
        if (needh) {
          const uint32_t fin = __ballot_sync(0xFFFFFFFFu, (uint32_t)(v >> 32) != NOHEAD);
          if (fin) {
            ch = __shfl_sync(0xFFFFFFFFu, (uint32_t)(v >> 32), __ffs(fin) - 1);
            needh = false;
          }
        }
        base -= 32;
      }
      if (lane == 0 && (flagf == 1u || flagh == 1u))  // forward the carry for the component(s) I have no head for
        st_relaxed_u64(tstate + tile, ((unsigned long long)(flagh == 1u ? ch : pubh) << 32) |
                                          (unsigned long long)(flagf == 1u ? cf : pubf));
    }
    if (lane == 0) {
      s_cf = cf;
      s_ch = ch;
      // head flag of the first record of the next tile (for the singleton test of my last record)
      uint32_t nh = 1u;
      const uint32_t jn = tile_base + TILE;
      if (jn < m) {
        const KeyT nk = keys[jn];
        const KeyT lk = s_lastkey[BLOCK - 1];
        const uint32_t ls = ROUND0 ? s_lastshort[BLOCK - 1] : 0u;
        nh = (nk != lk || ls) ? 1u : 0u;
      }
      s_firsthead[BLOCK] = nh;
    }
  }
  __syncthreads();
  exf = max(exf, s_cf);
  exh = max(exh, s_ch);
  const uint32_t nexthead_thread = s_firsthead[tid + 1];

  const bool bucketed = rp.nbuckets > 1;
  uint32_t live = 0, livemask = 0, gmax = 0, nrv[IPT];
  uint32_t wrmask = 0, bpos[IPT];
  uint32_t anymask = 0;  // records whose rank word changed or became final (whatever their id window)
  uint32_t embits = 0, ew0 = 0, ew1 = 0;  // ROUND0: the BWT bytes of my eight (consecutive) sorted positions
  uint32_t sabits = 0;                    // SA && ROUND0: which of them are final (their SA entries leave as whole words)
#pragma unroll
  for (int k = 0; k < IPT; ++k) {
    const uint32_t j = j0 + k;
    nrv[k] = 0;
    bpos[k] = 0;
    if (j < m) {
      const uint32_t HF = max(lf[k], exf) - 1u;  // >= 0: record 0 is always a head
      const bool hf = (headfull >> k) & 1u;
      const bool nh = (k == IPT - 1) ? (nexthead_thread != 0) : ((headfull >> (k + 1)) & 1u);
      const bool single = hf && nh;
      uint32_t nr;
      bool changed;
      if (ROUND0) {
        nr = HF;
        changed = true;
      } else {
        const uint32_t HH = max(lh[k], exh) - 1u;
        nr = (((uint32_t)(key[k] >> rp.lo_bits) << 1) | ((lowbits >> k) & 1u)) + (HF - HH);
        changed = (HF != HH);
      }
      const bool in_win = (id[k] >= rp.win_lo) && (id[k] < rp.win_hi);
      const bool emit_here = rp.emit == 1u || (rp.emit == 0u && in_win);
      if (single && emit_here && !owns_hole(ep, id[k]) && !(LAZY && rp.lazy == 2u)) {  // emit L[nr] = T[id-1]
        uint8_t ch;
        if (ROUND0 && rp.packed) ch = s_dec[((k < 4 ? pc0 >> (8 * k) : pc1 >> (8 * (k - 4)))) & 0xFFu];
        else ch = ep.text[id[k] - 1];
        if (ROUND0) {  // nr == j: collected, stored after the loop
          embits |= 1u << k;
          if (k < 4) ew0 |= (uint32_t)ch << (8 * k); else ew1 |= (uint32_t)ch << (8 * (k - 4));
        } else {
          emit_bwt(ep, nr, ch);
        }
      }
      // SA[nr] = id, under the same "emitted by this launch" rule as the BWT byte, but for suffix 0 too
      if (SA && single && emit_here && !(LAZY && rp.lazy == 2u)) {
        if (ROUND0) sabits |= 1u << k;
        else ep.sa[nr] = (int32_t)id[k];
      }
      if (single) nr |= RANK_DONE;
      else if (sp.enable) { ++live; livemask |= 1u << k; gmax = max(gmax, j - HF + 1u); }
      nrv[k] = nr;
      if (!ROUND0 && (changed || single)) anymask |= 1u << k;  // (round 0: every rank is new)
      bool wr = in_win && (changed || single);
      if (LAZY && rp.lazy) {
        const bool isshort = id[k] >= rp.short_thresh;
        if (rp.lazy == 1u) {
          wr = in_win && (!single || isshort);  // a singleton's rank is its sorted position: not stored (rank_lookup)
          if (wr) atomicOr(&rp.livebits[id[k] >> 5], 1u << (id[k] & 31u));
          // first sorted position of every key prefix
          const uint32_t pfx = (uint32_t)(key[k] >> rp.tshift);
          const bool firstrec = (k == 0 && !has_prev);
          const uint32_t ppfx = firstrec ? 0xFFFFFFFFu : (uint32_t)(((k == 0) ? prevkey : key[k - 1]) >> rp.tshift);
          if (firstrec || pfx != ppfx) rp.ktab[pfx] = j;
        } else {
          wr = in_win && single && !isshort;    // materialise the singletons (everything else is in place)
        }
      }
      if (wr) {
        if (bucketed) {
          const uint32_t b = min(__umulhi(id[k], rp.bucket_magic), rp.nbuckets - 1u);
          if (rp.direct0 && b == 0u) {
            rank[id[k]] = nr;
          } else {
            bpos[k] = atomicAdd(&s_bcnt[b], 1u);
            wrmask |= 1u << k;
          }
        } else {
          rank[id[k]] = nr;
        }
      }
    }
  }
  if (ROUND0 && embits) {
    // A singleton's rank is its sorted position, so my eight records are the output bytes j0 .. j0+7: one 8-byte (or
    // 4-byte) store when all of them are emitted, instead of byte stores that touch eight sectors per warp instruction.
    // `plain`: none of the eight positions is the parked last byte of a block (emit_bwt) and the buffer is aligned.
    bool plain = (reinterpret_cast<uintptr_t>(ep.out) & 7u) == 0u;
    if (ep.nblocks <= 1u) {
      plain = plain && !(ep.block_mode && j0 + 8u > ep.N - 1u);
    } else {
      const uint32_t kb = j0 / ep.stride;
      const uint32_t last = ((kb + 1u == ep.nblocks) ? ep.N : (kb + 1u) * ep.stride) - 1u;
      plain = plain && (j0 + 7u < last);
    }
    if (plain && embits == 0xFFu) {
      *reinterpret_cast<uint2*>(ep.out + j0) = make_uint2(ew0, ew1);
    } else {
      if (plain && (embits & 0xFu) == 0xFu) {
        *reinterpret_cast<uint32_t*>(ep.out + j0) = ew0;
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if ((embits >> k) & 1u) emit_bwt(ep, j0 + k, (uint8_t)(ew0 >> (8 * k)));
      }
      if (plain && (embits & 0xF0u) == 0xF0u) {
        *reinterpret_cast<uint32_t*>(ep.out + j0 + 4) = ew1;
      } else {
#pragma unroll
        for (int k = 4; k < 8; ++k)
          if ((embits >> k) & 1u) emit_bwt(ep, j0 + k, (uint8_t)(ew1 >> (8 * (k - 4))));
      }
    }
  }
  if (SA && ROUND0 && sabits) {  // the same eight positions: SA[j0 + k] = id[k], one 16-byte store per four final records
    int32_t* ps = ep.sa + j0;
    const bool al = (reinterpret_cast<uintptr_t>(ep.sa) & 15u) == 0u;  // (j0 % 8 == 0)
    if (al && (sabits & 0xFu) == 0xFu) {
      *reinterpret_cast<int4*>(ps) = make_int4((int)id[0], (int)id[1], (int)id[2], (int)id[3]);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if ((sabits >> k) & 1u) ps[k] = (int32_t)id[k];
    }
    if (al && (sabits & 0xF0u) == 0xF0u) {
      *reinterpret_cast<int4*>(ps + 4) = make_int4((int)id[4], (int)id[5], (int)id[6], (int)id[7]);
    } else {
#pragma unroll
      for (int k = 4; k < 8; ++k)
        if ((sabits >> k) & 1u) ps[k] = (int32_t)id[k];
    }
  }
  if (rp.nr_out) {
    uint32_t v[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) v[k] = (ROUND0 || ((anymask >> k) & 1u)) ? nrv[k] : 0xFFFFFFFFu;
    if (tile_base + TILE <= m) {
      uint4* po = reinterpret_cast<uint4*>(rp.nr_out + j0);  // j0 % 8 == 0, buffer 256-byte aligned
      __stcs(po, make_uint4(v[0], v[1], v[2], v[3]));
      __stcs(po + 1, make_uint4(v[4], v[5], v[6], v[7]));
    } else {
#pragma unroll
      for (int k = 0; k < IPT; ++k)
        if (j0 + k < m) rp.nr_out[j0 + k] = v[k];
    }
  }
  if (bucketed) {
    __syncthreads();
    if (tid == 0) {  // exclusive starts of the buckets inside this tile's slot
      uint32_t acc = 0;
      uint32_t* wo = sp.tile_woff + (size_t)tile * (rp.nbuckets + 1u);
      for (uint32_t b = 0; b < rp.nbuckets; ++b) {
        const uint32_t c = s_bcnt[b];
        s_bcnt[b] = acc;
        wo[b] = acc;
        acc += c;
      }
      wo[rp.nbuckets] = acc;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      if ((wrmask >> k) & 1u) {
        const uint32_t b = min(__umulhi(id[k], rp.bucket_magic), rp.nbuckets - 1u);
        const uint32_t dst = tile_base + s_bcnt[b] + bpos[k];
        sp.sc_id[dst] = id[k];
        sp.sc_nr[dst] = nrv[k];
      }
    }
  }
  if (!sp.enable) return;
  // ---- stage the records that stay live: (new rank, id) in sorted order at the start of this tile's slot
  uint32_t inc = live;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
    if (lane >= o) inc += t;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) gmax = max(gmax, __shfl_xor_sync(0xFFFFFFFFu, gmax, o));
  __syncthreads();  // s_wf is free again
  if (lane == 31) s_wf[warp] = inc;
  if (lane == 0 && gmax) atomicMax(&ctrl[CTR_MAXGROUP], gmax);
  __syncthreads();
  uint32_t woff = 0, total = 0;
#pragma unroll
  for (int w = 0; w < WARPS; ++w) {
    const uint32_t t = s_wf[w];
    if (w < warp) woff += t;
    total += t;
  }
  if (tid == 0) {
    sp.tile_cnt[tile] = total;
    if (total) atomicAdd(&ctrl[CTR_LIVE], total);
  }
  if (live) {
    uint32_t pos = tile_base + woff + inc - live;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      if ((livemask >> k) & 1u) {
        sp.stage_nr[pos] = nrv[k];
        sp.stage_id[pos] = id[k];
        ++pos;
      }
    }
  }
}

// k_scatter_bucket — rank[id] = nr for the staged records of ONE id bucket (all tiles).  One warp per tile
// segment; the bucket's slice of rank[] (<= ~72 MB) stays L2-resident, so the random 4-byte writes never pay a
// DRAM sector fill + write-back, and — unlike re-running k_rerank once per window — every record is read once.
// k_scatter_window — rank[id] = new rank for the records whose id lies in [win_lo, win_hi), from the sorted ids and the
// rank words k_rerank left beside them (RerankParams::nr_out).  Sequential 128-bit reads, L2-resident random writes.
__global__ void __launch_bounds__(256) k_scatter_window(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ nrw,
                                                        uint32_t m, uint32_t id_mask, uint32_t win_lo, uint32_t win_hi,
                                                        uint32_t* __restrict__ rank, const uint32_t* __restrict__ ctrl) {
  if (ctrl[CTR_ERR]) return;  // sticky error: the rank words may be incomplete
  const uint32_t quads = m >> 2;
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += gridDim.x * blockDim.x) {
    const uint4 i4 = __ldcs(reinterpret_cast<const uint4*>(idx) + q);
    const uint4 n4 = __ldcs(reinterpret_cast<const uint4*>(nrw) + q);
    const uint32_t ii[4] = {i4.x & id_mask, i4.y & id_mask, i4.z & id_mask, i4.w & id_mask};
    const uint32_t nn[4] = {n4.x, n4.y, n4.z, n4.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (nn[k] != 0xFFFFFFFFu && ii[k] >= win_lo && ii[k] < win_hi) rank[ii[k]] = nn[k];
  }
  if (blockIdx.x == 0 && threadIdx.x < (m & 3u)) {
    const uint32_t j = (m & ~3u) + threadIdx.x;
    const uint32_t i = idx[j] & id_mask, n = nrw[j];
    if (n != 0xFFFFFFFFu && i >= win_lo && i < win_hi) rank[i] = n;
  }
}

__global__ void __launch_bounds__(256) k_scatter_bucket(const uint32_t* __restrict__ sc_id, const uint32_t* __restrict__ sc_nr,
                                                        const uint32_t* __restrict__ tile_woff, uint32_t ntiles,
                                                        uint32_t nbuckets, uint32_t b, uint32_t tile_records,
                                                        uint32_t* __restrict__ rank, const uint32_t* __restrict__ ctrl) {
  if (ctrl[CTR_ERR]) return;  // sticky error: the staged pairs may be incomplete
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t nw = gridDim.x * (blockDim.x >> 5);
  for (uint32_t tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); tile < ntiles; tile += nw) {
    const uint32_t* wo = tile_woff + (size_t)tile * (nbuckets + 1u);
    const uint32_t lo = wo[b], hi = wo[b + 1];
    const size_t base = (size_t)tile * tile_records;
#pragma unroll 4
    for (uint32_t t = lo + lane; t < hi; t += 32) rank[__ldcs(sc_id + base + t)] = __ldcs(sc_nr + base + t);
  }
}

// =====================================================================================================
// Device-side round control ("ladder").  After a sort round (round 0 or a global radix round) the host does NOT
// read the live count back to decide what comes next: it enqueues the whole remaining sequence — live lists,
// a few segmented rounds, the single-CTA tail, k_finish, the result copies — and every kernel decides from this
// device-resident state whether it has work (k_commit_* update it between the kernels).  A block whose later rounds
// are all sort-free therefore needs ONE host synchronisation after round 0 instead of one per round; only when the
// ladder ends with suffixes still live (large groups: a global radix round is needed, or more segmented rounds than
// were enqueued) does the host step in again with the state it reads back.
// =====================================================================================================
constexpr int LADDER_LOG = 40;  // == BWTC_CUDA_MAX_ROUNDS
constexpr int SEG_T = 1920, SEG_CAP = 2048, SEG_MAXGROUP = 128;
constexpr int SMALL_MAX = 2048;
struct LadderState {
  uint32_t m;         // live records (suffixes in non-singleton groups)
  uint32_t maxgroup;  // largest group among them
  uint32_t h;         // prefix length every group agrees on (doubles per round, capped at 0x7FFFFFFF)
  uint32_t sel;       // pool indices of the rank-ordered (rank, id) lists of the live records: nr | id << 4
  uint32_t nlog;      // rounds logged below
  uint32_t lists;     // != 0: the lists at `sel` are valid
  uint32_t err;       // copy of ctrl[CTR_ERR] taken by k_finish (so one D2H brings everything back)
  uint32_t nruns;     // run statistics (k_run_emit): maximal runs of equal bytes in the finished output
  uint32_t pad2[4];
  uint32_t log_m[LADDER_LOG];     // records processed by ladder round i
  uint32_t log_kind[LADDER_LOG];  // 1 = segmented round, 2 = tail (k_small_rounds: all remaining rounds)
  uint32_t log_h[LADDER_LOG];
};
// The six u32[N] work arrays (halves of the two key buffers, the two id buffers) the lists rotate through.
struct PoolPtrs { uint32_t* p[6]; };

__device__ __forceinline__ bool ladder_wants_seg(const LadderState& st) {
  return st.lists && st.m > (uint32_t)SMALL_MAX && st.maxgroup <= (uint32_t)SEG_MAXGROUP;
}
__device__ __forceinline__ bool ladder_wants_lists(uint32_t m, uint32_t maxgroup) {
  return m != 0u && (m <= (uint32_t)SMALL_MAX || maxgroup <= (uint32_t)SEG_MAXGROUP);
}
// out_nr, out_id, upd_a, upd_b = the four pool arrays not holding the current lists, in index order
__device__ __forceinline__ void ladder_free_slots(uint32_t sel, int* f) {
  const int a = (int)(sel & 15u), b = (int)(sel >> 4);
  int nf = 0;
#pragma unroll
  for (int q = 0; q < 6; ++q)
    if (q != a && q != b && nf < 4) f[nf++] = q;
}

// After a sort round: take the re-rank's totals, name the place the lists WILL be in (k_gather_chunks builds them
// only if the next step consumes them), clear the accumulators for the segmented rounds.
__global__ void k_commit_sort(LadderState* st, uint32_t* ctrl, uint32_t h_new, uint32_t sel_lists, uint32_t expect_cursor,
                              uint32_t will_build_lists, uint32_t list_capacity) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  // k_build_keys must have emitted exactly the records the previous round left live (0xFFFFFFFF: no such check)
  if (expect_cursor != 0xFFFFFFFFu && ctrl[CTR_CURSOR] != expect_cursor && !ctrl[CTR_ERR]) ctrl[CTR_ERR] = 5u;
  const uint32_t m = ctrl[CTR_LIVE], g = ctrl[CTR_MAXGROUP];
  st->m = m;
  st->maxgroup = g;
  st->h = h_new;
  st->sel = sel_lists;
  // (k_gather_chunks follows only if will_build_lists; lazy ranks keep the lists in a smaller pool: if the live records do
  // not fit, nothing is built and the host falls back to the full path)
  st->lists = (will_build_lists && m <= list_capacity && ladder_wants_lists(m, g)) ? 1u : 0u;
  ctrl[CTR_LIVE] = 0;
  ctrl[CTR_MAXGROUP] = 0;
  ctrl[CTR_UPD] = 0;
}

// The host built the lists unconditionally (make_lists(false)) behind a lean chunk: tell the ladder kernels.
__global__ void k_mark_lists(LadderState* st, uint32_t sel_lists) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  st->sel = sel_lists;
  st->lists = 1u;
}

// After k_seg_round + k_apply_ranks.
__global__ void k_commit_seg(LadderState* st, uint32_t* ctrl) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (!ladder_wants_seg(*st) || ctrl[CTR_ERR]) return;  // the round did not run
  const uint32_t i = st->nlog;
  if (i < (uint32_t)LADDER_LOG) { st->log_m[i] = st->m; st->log_kind[i] = 1u; st->log_h[i] = st->h; st->nlog = i + 1u; }
  int f[4];
  ladder_free_slots(st->sel, f);
  st->sel = (uint32_t)f[0] | ((uint32_t)f[1] << 4);
  st->m = ctrl[CTR_LIVE];
  st->maxgroup = ctrl[CTR_MAXGROUP];
  st->h = st->h >= 0x40000000u ? 0x7FFFFFFFu : st->h * 2u;
  ctrl[CTR_LIVE] = 0;
  ctrl[CTR_MAXGROUP] = 0;
  ctrl[CTR_UPD] = 0;
}

// k_scan_tile_counts (one CTA): exclusive prefix of the per-tile live counts.  k_gather_chunks: tile t copies its
// staged chunk to out[excl[t] ..) — the concatenation keeps the sorted order, so groups stay contiguous.
__global__ void __launch_bounds__(1024) k_scan_tile_counts(const uint32_t* __restrict__ cnt, uint32_t* __restrict__ excl,
                                                           uint32_t ntiles) {
  constexpr int PER = 16;  // counts per thread and sweep: 16 independent loads in flight, one CTA scan per 16384 tiles
  __shared__ uint32_t s_w[32];
  __shared__ uint32_t s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < ntiles; base += 1024 * PER) {
    const uint32_t i0 = base + (uint32_t)tid * PER;
    uint32_t v[PER];
#pragma unroll
    for (int k = 0; k < PER; ++k) v[k] = (i0 + k < ntiles) ? cnt[i0 + k] : 0u;
    uint32_t sum = 0;
#pragma unroll
    for (int k = 0; k < PER; ++k) sum += v[k];
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    uint32_t woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 32; ++w) { const uint32_t t = s_w[w]; if (w < warp) woff += t; total += t; }
    const uint32_t carry = s_carry;
    uint32_t run = carry + woff + inc - sum;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
      if (i0 + k < ntiles) excl[i0 + k] = run;
      run += v[k];
    }
    __syncthreads();
    if (tid == 0) s_carry = carry + total;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) k_gather_chunks(const uint32_t* __restrict__ stage_nr,
                                                       const uint32_t* __restrict__ stage_id,
                                                       const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ excl,
                                                       uint32_t tile_records, uint32_t* __restrict__ out_nr,
                                                       uint32_t* __restrict__ out_id,
                                                       const LadderState* __restrict__ st, const uint32_t* __restrict__ ctrl) {
  // st != nullptr: speculative launch — only if the next step consumes the lists (k_commit_sort decided)
  const uint32_t tile = blockIdx.x;
  const uint32_t wanted = st ? st->lists : 1u, err = ctrl[CTR_ERR];  // (all four loads are issued before the first branch)
  const uint32_t c = cnt[tile], dst = excl[tile];
  if (!wanted || err) return;
  const size_t src = (size_t)tile * tile_records;
  for (uint32_t t = threadIdx.x; t < c; t += blockDim.x) {
    out_nr[dst + t] = stage_nr[src + t];
    out_id[dst + t] = stage_id[src + t];
  }
}

// =====================================================================================================
// k_build_from_list — doubling-round key build for rounds with few live suffixes: the ids come from the compact
// list built from k_rerank's staging (no scan over all N ranks); two rank gathers per record.  Same key layout and fused
// histograms as k_build_keys.
// =====================================================================================================
__global__ void __launch_bounds__(256) k_build_from_list(const uint32_t* __restrict__ list, uint32_t m,
                                                         const uint32_t* __restrict__ rank, uint32_t N, uint32_t h,
                                                         int lo_bits, unsigned long long* __restrict__ keys,
                                                         uint32_t* __restrict__ idx, uint32_t* __restrict__ hist,
                                                         int npass, const uint32_t* __restrict__ ctrl, uint32_t rb) {
  __shared__ uint32_t s_hist[8 * 512];
  const int tid = threadIdx.x;
  const uint32_t dmask = (1u << rb) - 1u;
  if (ctrl[CTR_ERR]) return;
#pragma unroll
  for (int p = 0; p < 16; ++p) s_hist[p * 256 + tid] = 0;
  __syncthreads();
  for (uint32_t j = blockIdx.x * blockDim.x + tid; j < m; j += gridDim.x * blockDim.x) {
    const uint32_t i = list[j];
    const uint32_t r = rank[i] & RANK_MASK;
    const uint32_t r2 = (h < N - i) ? ((rank[i + h] & RANK_MASK) + 1u) : 0u;
    const unsigned long long key = ((unsigned long long)(r >> 1) << lo_bits) | (unsigned long long)r2;  // see k_build_keys
    keys[j] = key;
    idx[j] = i | ((r & 1u) << 31);
    for (int p = 0; p < npass; ++p) atomicAdd(&s_hist[(p << rb) + ((uint32_t)(key >> (rb * p)) & dmask)], 1u);
  }
  __syncthreads();
  for (int p = 0; p < npass; ++p)
    for (uint32_t e = tid; e <= dmask; e += 256) {
      const uint32_t v = s_hist[(p << rb) + e];
      if (v) atomicAdd(&hist[(p << rb) + e], v);
    }
}

// =====================================================================================================
// k_seg_round — one doubling round WITHOUT a global sort, for rounds whose groups are all small.
// After any round the still-live records sit in rank order with every group contiguous, so the next round only
// has to order each group by rank[i+h]: a tile of ~1920 records, extended to the next group boundary on both
// sides (groups are <= SEG_MAXGROUP long, checked by the host from ctrl[CTR_MAXGROUP]), has each of its groups
// ordered by (old rank, rank[i+h]) by counting inside the group in shared memory, is re-ranked, its new singletons are emitted, and
// the records still tied are appended — whole groups at a time, in order — as the input of the next round.
// One kernel replaces key build + 7 digit passes + re-rank (~0.45 ms for the 2.6 M live suffixes of the Markov
// block's second round).  Input may contain holes (RANK_DONE records of the previous global sort).
// Replaces tr_introsort over small groups (trsort.c:327-552).
// =====================================================================================================
#ifndef BWTC_SEG_MINB
#define BWTC_SEG_MINB 4
#endif

// Persistent grid: tile t = blockIdx.x, blockIdx.x + gridDim.x, ... while t * SEG_T < m (m is read from the
// device-side LadderState, so the host can enqueue the round before it knows how many suffixes are live).
#ifndef BWTC_SEG_MINB_LAZY
#define BWTC_SEG_MINB_LAZY 4  // (3 CTAs/SM with 80 registers measured the same)
#endif
template <bool LAZY, bool SA = false>
__global__ void __launch_bounds__(256, LAZY ? BWTC_SEG_MINB_LAZY : BWTC_SEG_MINB) k_seg_round(const LadderState* __restrict__ st, PoolPtrs pool,
                                                   const uint32_t* __restrict__ rank, uint32_t N, EmitParams ep,
                                                   uint32_t* __restrict__ ctrl, const LookupParams* __restrict__ lkp) {
  constexpr int IPT = SEG_CAP / 256;
  __shared__ unsigned long long s_key[SEG_CAP];
  __shared__ uint32_t s_id[SEG_CAP];
  __shared__ unsigned long long s_k0[LAZY ? SEG_CAP : 1];  // lazy: round-0 key of suffix i+h (first part of cmp(i+h))
  __shared__ uint32_t s_wa[8], s_wb[8];
  __shared__ uint32_t s_start, s_end, s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t m_in = st->m, h = st->h, st_maxgroup = st->maxgroup, st_lists = st->lists, err = ctrl[CTR_ERR];
  if (!(st_lists && m_in > (uint32_t)SMALL_MAX && st_maxgroup <= (uint32_t)SEG_MAXGROUP) || err) return;  // ladder_wants_seg
  // the six list pointers live in shared memory (they would cost 12 registers across the tile loop)
  __shared__ uint32_t* s_ptr[6];  // [0] nr_in [1] id_in [2] nr_out [3] id_out [4] upd_id [5] upd_nr
  if (tid == 0) {
    int fslot[4];
    ladder_free_slots(st->sel, fslot);
    s_ptr[0] = pool.p[st->sel & 15u];
    s_ptr[1] = pool.p[st->sel >> 4];
    for (int q = 0; q < 4; ++q) s_ptr[2 + q] = pool.p[fslot[q]];
  }
#define nr_in (static_cast<const uint32_t*>(s_ptr[0]))
#define id_in (static_cast<const uint32_t*>(s_ptr[1]))
#define nr_out (s_ptr[2])
#define id_out (s_ptr[3])
#define upd_id (s_ptr[4])
#define upd_nr (s_ptr[5])
  for (uint32_t a = blockIdx.x * (uint32_t)SEG_T; a < m_in; a += gridDim.x * (uint32_t)SEG_T) {
  __syncthreads();  // shared memory of the previous tile is free (first trip: s_ptr is visible)
  const uint32_t b = (m_in - a > (uint32_t)SEG_T) ? a + SEG_T : m_in;
  if (tid == 0) { s_start = 0xFFFFFFFFu; s_end = (b >= m_in) ? m_in : 0xFFFFFFFFu; }
  __syncthreads();
  // ---- extend the tile to group boundaries: first group head at or after a, first group head at or after b
  for (uint32_t t = tid; t <= (uint32_t)SEG_MAXGROUP; t += 256) {
    const uint32_t ja = a + t;
    if (ja < m_in) {
      if (ja == 0 || nr_in[ja] != nr_in[ja - 1]) atomicMin(&s_start, ja);
    } else if (ja == m_in) {
      atomicMin(&s_start, m_in);
    }
    const uint32_t jb = b + t;
    if (b < m_in) {
      if (jb < m_in) {
        if (nr_in[jb] != nr_in[jb - 1]) atomicMin(&s_end, jb);
      } else if (jb == m_in) {
        atomicMin(&s_end, m_in);
      }
    }
  }
  __syncthreads();
  const uint32_t start = s_start, end = s_end;
  if (start == 0xFFFFFFFFu || end == 0xFFFFFFFFu || (start < end && end - start > (uint32_t)SEG_CAP)) {
    if (tid == 0) atomicExch(&ctrl[CTR_ERR], 4u);  // a group longer than SEG_MAXGROUP: this path must not be picked
    continue;
  }
  if (start >= end) continue;
  // ---- load my records (thread-blocked, order preserved), drop the holes, build (old rank, rank[i+h]) keys
  uint32_t myid[IPT], mynr[IPT];
  uint32_t livemask = 0;
#pragma unroll
  for (int k = 0; k < IPT; ++k) {
    const uint32_t j = start + tid * IPT + k;
    mynr[k] = RANK_DONE;
    myid[k] = 0;
    if (j < end) { mynr[k] = nr_in[j]; myid[k] = id_in[j]; }
    if (!(mynr[k] & RANK_DONE)) livemask |= 1u << k;
  }
  uint32_t cnt = __popc(livemask), inc = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_wa[warp] = inc;
  __syncthreads();
  uint32_t woff = 0, L = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) { const uint32_t t = s_wa[w]; if (w < warp) woff += t; L += t; }
  if constexpr (!LAZY) {
    uint32_t lo[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {  // independent gathers first (all in flight together), shared-memory writes after
      lo[k] = 0;
      if (((livemask >> k) & 1u) && h < N - myid[k]) lo[k] = (rank[myid[k] + h] & RANK_MASK) + 1u;
    }
    uint32_t pos = woff + inc - cnt;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      if ((livemask >> k) & 1u) {
        s_key[pos] = ((unsigned long long)mynr[k] << 32) | lo[k];
        s_id[pos] = myid[k];
        ++pos;
      }
    }
  } else {
    // Lazy ranks (DESIGN.md §3.9): the integer rank of i+h is not needed, only the order and equality of the members of a
    // group, and cmp(j) = (round-0 key of j, livebits(j) ? rank[j] + 1 : 0xFFFFFFFF) gives both — no search.  A suffix
    // with i+h >= N gets (0, 0), below every real cmp (those have a second part >= 1), as the 0 of the full path.
    uint32_t pos = woff + inc - cnt;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      if ((livemask >> k) & 1u) {
        unsigned long long k0 = 0;
        uint32_t lo = 0;
        if (h < N - myid[k]) {
          const uint32_t j = myid[k] + h;
          const uint32_t lw = lkp->livebits[j >> 5];  // (issued before the key's text loads)
          k0 = round0_key(*lkp, j);
          lo = ((lw >> (j & 31u)) & 1u) ? (rank[j] & RANK_MASK) + 1u : 0xFFFFFFFFu;
        }
        s_key[pos] = ((unsigned long long)mynr[k] << 32) | lo;
        s_k0[pos] = k0;
        s_id[pos] = myid[k];
        ++pos;
      }
    }
  }
  __syncthreads();
  if (L == 0) continue;
  const uint32_t P = L;
  // ---- order every group by counting: the records are already grouped by old rank, groups are short
  // (<= SEG_MAXGROUP), so each record just counts the members of its own group that precede it.  No sorting
  // network: a full bitonic sort of the tile was measured 8x slower (374 us for 2.6 M records).
  {
    unsigned long long kreg[IPT];
    uint32_t ireg[IPT], npos[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      // striped (record tid + 256k): the members of a long group are spread over many threads and the lanes of a
      // warp walk the same group together (broadcast reads), instead of one thread owning 8 members of it
      const uint32_t j = (uint32_t)tid + 256u * k;
      npos[k] = 0xFFFFFFFFu;
      if (j < L) {
        kreg[k] = s_key[j];
        ireg[k] = s_id[j];
        const uint32_t g = (uint32_t)(kreg[k] >> 32);
        uint32_t cntb = 0, gs = j;
        if constexpr (!LAZY) {
          for (uint32_t q = j; q-- > 0;) {
            const unsigned long long kq = s_key[q];
            if ((uint32_t)(kq >> 32) != g) break;
            cntb += (kq <= kreg[k]) ? 1u : 0u;
            gs = q;
          }
          for (uint32_t q = j + 1; q < L; ++q) {
            const unsigned long long kq = s_key[q];
            if ((uint32_t)(kq >> 32) != g) break;
            cntb += (kq < kreg[k]) ? 1u : 0u;
          }
        } else {
          // order by cmp = (s_k0, low word of s_key).  My key for the re-rank below becomes (old rank, number of group
          // members with a smaller cmp): it orders and ties exactly as cmp does
          const unsigned long long k0 = s_k0[j];
          const uint32_t lo = (uint32_t)kreg[k];
          uint32_t nlt = 0;
          for (uint32_t q = j; q-- > 0;) {
            const unsigned long long kq = s_key[q];
            if ((uint32_t)(kq >> 32) != g) break;
            const unsigned long long k0q = s_k0[q];
            const bool lt = k0q < k0 || (k0q == k0 && (uint32_t)kq < lo);
            nlt += lt ? 1u : 0u;
            cntb += (lt || (k0q == k0 && (uint32_t)kq == lo)) ? 1u : 0u;
            gs = q;
          }
          for (uint32_t q = j + 1; q < L; ++q) {
            const unsigned long long kq = s_key[q];
            if ((uint32_t)(kq >> 32) != g) break;
            const unsigned long long k0q = s_k0[q];
            const bool lt = k0q < k0 || (k0q == k0 && (uint32_t)kq < lo);
            nlt += lt ? 1u : 0u;
            cntb += lt ? 1u : 0u;
          }
          kreg[k] = ((unsigned long long)g << 32) | nlt;
        }
        npos[k] = gs + cntb;
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      if (npos[k] != 0xFFFFFFFFu) {
        s_key[npos[k]] = kreg[k];
        s_id[npos[k]] = ireg[k];
      }
    }
    __syncthreads();
  }
  // ---- re-rank inside the tile (it starts and ends on group boundaries: no carry from other tiles)
  unsigned long long key[IPT];
  uint32_t runf = 0, runh = 0, lf[IPT], lh[IPT], hfmask = 0;
  const uint32_t j0 = tid * IPT;
#pragma unroll
  for (int k = 0; k < IPT; ++k) {
    const uint32_t j = j0 + k;
    key[k] = (j < P) ? s_key[j] : ~0ull;
    myid[k] = (j < P) ? s_id[j] : 0u;
    const unsigned long long pk = (j > 0 && j <= P) ? s_key[j - 1] : 0ull;
    const bool hf = (j == 0) || (j >= L) || (key[k] != pk);
    const bool hh = (j == 0) || (j >= L) || ((key[k] >> 32) != (pk >> 32));
    if (hf) { hfmask |= 1u << k; runf = j + 1; }
    if (hh) runh = j + 1;
    lf[k] = runf;
    lh[k] = runh;
  }
  const unsigned long long nextkey = (j0 + IPT < P) ? s_key[j0 + IPT] : ~0ull;
  uint32_t incf = runf, inch = runh;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t tf = __shfl_up_sync(0xFFFFFFFFu, incf, o), th = __shfl_up_sync(0xFFFFFFFFu, inch, o);
    if (lane >= o) { incf = max(incf, tf); inch = max(inch, th); }
  }
  uint32_t exf = __shfl_up_sync(0xFFFFFFFFu, incf, 1), exh = __shfl_up_sync(0xFFFFFFFFu, inch, 1);
  if (lane == 0) { exf = 0; exh = 0; }
  __syncthreads();  // everyone has read s_key / s_id into registers
  if (lane == 31) { s_wa[warp] = incf; s_wb[warp] = inch; }
  __syncthreads();
  for (int w = 0; w < warp; ++w) { exf = max(exf, s_wa[w]); exh = max(exh, s_wb[w]); }
  // NOTE: rank[] is NOT written here.  Other CTAs are still reading rank[i+h] of this round; a half-refined
  // rank[] could order two members of one group by ranks of different generations.  Changed ranks go to an
  // update list that k_apply_ranks scatters after this kernel.
  uint32_t keep = 0, updm = 0, newnr[IPT], gmax = 0;
#pragma unroll
  for (int k = 0; k < IPT; ++k) {
    const uint32_t j = j0 + k;
    newnr[k] = 0;
    if (j < L) {
      const uint32_t HF = max(lf[k], exf) - 1u, HH = max(lh[k], exh) - 1u;
      const unsigned long long nk = (k == IPT - 1) ? nextkey : key[k + 1];
      const bool single = ((hfmask >> k) & 1u) && (j + 1 >= L || nk != key[k]);
      uint32_t nr = (uint32_t)(key[k] >> 32) + (HF - HH);
      if (single && !owns_hole(ep, myid[k])) emit_bwt(ep, nr, ep.text[myid[k] - 1]);
      if (SA && single) ep.sa[nr] = (int32_t)myid[k];
      if (single) nr |= RANK_DONE; else { keep |= 1u << k; gmax = max(gmax, j - HF + 1u); }
      newnr[k] = nr;
      if (single || HF != HH) updm |= 1u << k;
    }
  }
  // ---- append the records still tied (whole groups, in order) for the next round, and the rank updates
  cnt = __popc(keep);
  inc = cnt;
  const uint32_t ucnt = __popc(updm);
  uint32_t uinc = ucnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
    const uint32_t tu = __shfl_up_sync(0xFFFFFFFFu, uinc, o);
    if (lane >= o) { inc += t; uinc += tu; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) gmax = max(gmax, __shfl_xor_sync(0xFFFFFFFFu, gmax, o));
  __syncthreads();
  if (lane == 31) { s_wa[warp] = inc; s_wb[warp] = uinc; }
  if (lane == 0 && gmax) atomicMax(&ctrl[CTR_MAXGROUP], gmax);
  __syncthreads();
  woff = 0;
  uint32_t total = 0, uoff = 0, utotal = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    const uint32_t t = s_wa[w], tu = s_wb[w];
    if (w < warp) { woff += t; uoff += tu; }
    total += t;
    utotal += tu;
  }
  if (tid == 0) {
    s_base = total ? atomicAdd(&ctrl[CTR_LIVE], total) : 0u;
    s_start = utotal ? atomicAdd(&ctrl[CTR_UPD], utotal) : 0u;  // s_start is free again
  }
  __syncthreads();
  if (cnt) {
    uint32_t pos = s_base + woff + inc - cnt;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      if ((keep >> k) & 1u) {
        nr_out[pos] = newnr[k];
        id_out[pos] = myid[k];
        ++pos;
      }
    }
  }
  if (ucnt) {
    uint32_t pos = s_start + uoff + uinc - ucnt;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
      if ((updm >> k) & 1u) {
        upd_id[pos] = myid[k];
        upd_nr[pos] = newnr[k];
        ++pos;
      }
    }
  }
  }  // tile loop
#undef nr_in
#undef id_in
#undef nr_out
#undef id_out
#undef upd_id
#undef upd_nr
}

// k_apply_ranks — second half of a segmented round: rank[id] = new rank for every record whose rank changed or
// became final.  The count is read from ctrl[CTR_UPD] on the device (no host round trip in between).
__global__ void __launch_bounds__(256) k_apply_ranks(const LadderState* __restrict__ st, PoolPtrs pool,
                                                     const uint32_t* __restrict__ ctrl, uint32_t* __restrict__ rank) {
  const uint32_t st_m = st->m, st_maxgroup = st->maxgroup, st_lists = st->lists, err = ctrl[CTR_ERR];
  if (!(st_lists && st_m > (uint32_t)SMALL_MAX && st_maxgroup <= (uint32_t)SEG_MAXGROUP) || err) return;  // the round did not run
  int fslot[4];
  ladder_free_slots(st->sel, fslot);
  const uint32_t* __restrict__ upd_id = pool.p[fslot[2]];
  const uint32_t* __restrict__ upd_nr = pool.p[fslot[3]];
  const uint32_t n = ctrl[CTR_UPD];
  const uint32_t stride = gridDim.x * blockDim.x;
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  for (; j + 3 * stride < n; j += 4 * stride) {  // four independent (id, rank) loads and stores in flight per thread
    const uint32_t i0 = upd_id[j], i1 = upd_id[j + stride], i2 = upd_id[j + 2 * stride], i3 = upd_id[j + 3 * stride];
    const uint32_t r0 = upd_nr[j], r1 = upd_nr[j + stride], r2 = upd_nr[j + 2 * stride], r3 = upd_nr[j + 3 * stride];
    rank[i0] = r0; rank[i1] = r1; rank[i2] = r2; rank[i3] = r3;
  }
  for (; j < n; j += stride) rank[upd_id[j]] = upd_nr[j];
}

// =====================================================================================================
// k_small_rounds — finishes the refinement when at most SMALL_MAX suffixes are still live: ONE CTA runs all
// remaining doubling rounds (key build, bitonic sort in shared memory, re-rank, BWT emission, compaction)
// without returning to the host, instead of ~10 launch-latency-bound kernels per round.
// Replaces the tail of trsort's loop (trsort.c:563-585), where only a few groups are left.
// =====================================================================================================
template <bool SA = false>
__global__ void __launch_bounds__(1024) k_small_rounds(LadderState* st, PoolPtrs pool, uint32_t* rank,
                                                       uint32_t N, EmitParams ep, uint32_t* __restrict__ ctrl,
                                                       const LookupParams* __restrict__ lkp) {
  __shared__ unsigned long long s_key[SMALL_MAX];
  __shared__ uint32_t s_id[SMALL_MAX];
  __shared__ uint32_t s_a[32], s_b[32];
  __shared__ uint32_t s_m;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t m0 = st->m;
  if (!st->lists || m0 == 0u || m0 > (uint32_t)SMALL_MAX || ctrl[CTR_ERR]) return;  // not (yet) the tail
  const uint32_t* __restrict__ list = pool.p[st->sel >> 4];
  for (int j = tid; j < SMALL_MAX; j += 1024) s_id[j] = (j < (int)m0) ? list[j] : 0u;
  uint32_t m = m0;
  unsigned long long h = st->h;
  uint32_t iters = 0;
  __syncthreads();  // (also: everybody has read the state before thread 0 rewrites it below)
  if (tid == 0) {
    const uint32_t i = st->nlog;
    if (i < (uint32_t)LADDER_LOG) { st->log_m[i] = m0; st->log_kind[i] = 2u; st->log_h[i] = st->h; st->nlog = i + 1u; }
    st->m = 0;
    st->maxgroup = 0;
  }
  while (m > 0) {
    if (++iters > 64u) {  // cannot happen (h doubles past N); watchdog instead of a hang
      if (tid == 0) atomicExch(&ctrl[CTR_ERR], 3u);
      break;
    }
    uint32_t P = 2;  // sort width: next power of two >= m
    while (P < m) P <<= 1;
    for (uint32_t j = tid; j < P; j += 1024) {
      unsigned long long key = ~0ull;  // pads sort last
      if (j < m) {
        const uint32_t i = s_id[j];
        const uint32_t hi = rank[i] & RANK_MASK;  // (i is live: its rank is always stored)
        uint32_t lo = 0u;
        if (h < (unsigned long long)(N - i))
          lo = (lkp ? rank_lookup(*lkp, rank, i + (uint32_t)h) : (rank[i + (uint32_t)h] & RANK_MASK)) + 1u;
        key = ((unsigned long long)hi << 32) | lo;
      }
      s_key[j] = key;
    }
    __syncthreads();
    for (uint32_t k = 2; k <= P; k <<= 1) {
      for (uint32_t jj = k >> 1; jj > 0; jj >>= 1) {
        for (uint32_t t = tid; t < P; t += 1024) {
          const uint32_t x = t ^ jj;
          if (x > t) {
            const unsigned long long a = s_key[t], b = s_key[x];
            const bool up = ((t & k) == 0);
            if ((a > b) == up) {
              s_key[t] = b; s_key[x] = a;
              const uint32_t ia = s_id[t]; s_id[t] = s_id[x]; s_id[x] = ia;
            }
          }
        }
        __syncthreads();
      }
    }
    // re-rank: thread t owns sorted positions 2t and 2t+1
    unsigned long long key2[2];
    uint32_t id2[2], hf2[2], hh2[2];
    uint32_t runf = 0, runh = 0, lf2[2], lh2[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const uint32_t j = 2 * tid + q;
      key2[q] = (j < P) ? s_key[j] : ~0ull;
      id2[q] = (j < P) ? s_id[j] : 0u;
      const unsigned long long pk = (j > 0 && j <= P) ? s_key[j - 1] : 0ull;
      hf2[q] = (j == 0 || j >= m || key2[q] != pk) ? 1u : 0u;
      hh2[q] = (j == 0 || j >= m || (key2[q] >> 32) != (pk >> 32)) ? 1u : 0u;
      if (hf2[q]) runf = j + 1;
      if (hh2[q]) runh = j + 1;
      lf2[q] = runf;
      lh2[q] = runh;
    }
    const unsigned long long nextkey = (2 * tid + 2 < P) ? s_key[2 * tid + 2] : ~0ull;
    // CTA-wide exclusive max-scan of (runf, runh)
    uint32_t incf = runf, inch = runh;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t tf = __shfl_up_sync(0xFFFFFFFFu, incf, o), th = __shfl_up_sync(0xFFFFFFFFu, inch, o);
      if (lane >= o) { incf = max(incf, tf); inch = max(inch, th); }
    }
    uint32_t exf = __shfl_up_sync(0xFFFFFFFFu, incf, 1), exh = __shfl_up_sync(0xFFFFFFFFu, inch, 1);
    if (lane == 0) { exf = 0; exh = 0; }
    if (lane == 31) { s_a[warp] = incf; s_b[warp] = inch; }
    __syncthreads();
    for (int w = 0; w < warp; ++w) { exf = max(exf, s_a[w]); exh = max(exh, s_b[w]); }
    __syncthreads();
    uint32_t keep = 0;  // bit q: record stays live
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const uint32_t j = 2 * tid + q;
      if (j < m) {
        const uint32_t HF = max(lf2[q], exf) - 1u, HH = max(lh2[q], exh) - 1u;
        const unsigned long long nk = (q == 0) ? key2[1] : nextkey;
        const bool single = hf2[q] && (j + 1 >= m || nk != key2[q]);
        uint32_t nr = (uint32_t)(key2[q] >> 32) + (HF - HH);
        if (single && !owns_hole(ep, id2[q])) emit_bwt(ep, nr, ep.text[id2[q] - 1]);
        if (SA && single) ep.sa[nr] = (int32_t)id2[q];
        if (single) nr |= RANK_DONE; else keep |= 1u << q;
        if (single || HF != HH) rank[id2[q]] = nr;
      }
    }
    // compact the ids that stay live to the front of s_id
    const uint32_t cnt = __popc(keep);
    uint32_t inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) s_a[warp] = inc;
    __syncthreads();  // also: every thread holds its ids in registers, s_id may be overwritten
    uint32_t woff = 0, total = 0;
    for (int w = 0; w < 32; ++w) {
      const uint32_t t = s_a[w];
      if (w < warp) woff += t;
      total += t;
    }
    uint32_t pos = woff + inc - cnt;
#pragma unroll
    for (int q = 0; q < 2; ++q)
      if ((keep >> q) & 1u) s_id[pos++] = id2[q];
    if (tid == 0) s_m = total;
    __syncthreads();  // new list + rank[] updates visible to the whole CTA
    m = s_m;
    h = (h * 2 > 0x7FFFFFFFull) ? 0x7FFFFFFFull : h * 2;
  }
}


// =====================================================================================================
// k_copy_out — OPTIONAL (BWTC_D2H_KERNEL=1): the result copy to a PINNED host buffer done by SMs (plain stores through the
// unified address space) instead of the copy engine.  Background: device-to-host traffic at the rate the end-to-end path
// needs slows the kernels of all other streams by 12% (tests/gpu_dma_interference.py: 12.6 -> 11.0 GB/s device-resident;
// host-to-device copies: -1%).  This kernel was built to see whether the copy ENGINE is to blame: it is not — the same
// bytes written by 16 CTAs cost the same (e2e 10.76 vs 10.70 GB/s), more CTAs cost more.  Not the default.
// 16-byte accesses where both pointers allow it, bytes at the ragged ends.  Skips an unfinished block (st->m != 0).
// =====================================================================================================
__global__ void __launch_bounds__(256) k_copy_out(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, uint32_t n,
                                                  const LadderState* __restrict__ st, const uint32_t* __restrict__ ctrl) {
  if (st->m != 0u || ctrl[CTR_ERR]) return;
  const uintptr_t mis = (16u - (reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u;  // bytes until dst is 16-byte aligned
  const uint32_t head = mis < n ? (uint32_t)mis : n;
  const uint32_t tidg = blockIdx.x * blockDim.x + threadIdx.x, nthr = gridDim.x * blockDim.x;
  if (tidg < head) dst[tidg] = src[tidg];
  const uint32_t body = (n - head) / 16u;
  uint4* d4 = reinterpret_cast<uint4*>(dst + head);
  if (((reinterpret_cast<uintptr_t>(src) + head) & 15u) == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src + head);
    for (uint32_t i = tidg; i < body; i += nthr) d4[i] = s4[i];
  } else {
    for (uint32_t i = tidg; i < body; i += nthr) {
      const uint8_t* sp = src + head + (size_t)i * 16u;
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        w[k] = (uint32_t)sp[4 * k] | ((uint32_t)sp[4 * k + 1] << 8) | ((uint32_t)sp[4 * k + 2] << 16) | ((uint32_t)sp[4 * k + 3] << 24);
      d4[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
  const uint32_t done = head + body * 16u;
  if (tidg < n - done) dst[done + tidg] = src[done + tidg];
}

// =====================================================================================================
// k_finish — primary index + LFpowers + hole fill (the BWT bytes themselves are emitted by k_rerank as soon
// as a suffix becomes unique; see EmitParams).  rank[] is now the inverse suffix array.
//   block contract (BWTransform.cpp:52-64): out[0..n) = L[0..n) with out[pidx] = L[N-1] (hole fill);
//   raw contract   (divsufsort.c:506-512) : U[r] = L[r] for r != pidx, U[pidx] = T[pidx] ("untouched").
//   LFpowers[0] = pidx = rank[0]; LFpowers[j] = rank[N - j*(N/nLF)]     (divsufsort.c:337-338,350,381,390,500).
// Replaces construct_BWT / construct_BWT_orig (divsufsort.c:259-404) and the copy loop (:506-512).
// =====================================================================================================
__global__ void __launch_bounds__(256) k_finish(const uint32_t* __restrict__ rank, const uint8_t* __restrict__ text,
                                                uint32_t N, uint8_t* __restrict__ out, int block_mode,
                                                uint32_t* __restrict__ LF, uint32_t nLF,
                                                const uint32_t* __restrict__ lastch, LadderState* st,
                                                const uint32_t* __restrict__ ctrl, const LookupParams* __restrict__ lkp) {
  const uint32_t tid = threadIdx.x;
  const uint32_t err = ctrl[CTR_ERR];
  if (tid == 0) st->err = err;
  if (err || st->m != 0u) return;  // failed (rank[] is not trustworthy), or refinement not finished yet: the host
                                   // continues and launches k_finish again
  const uint32_t pidx = lkp ? rank_lookup(*lkp, rank, 0u) : (rank[0] & RANK_MASK);
  if (tid < nLF) {
    const uint32_t x = N / nLF;
    LF[tid] = (tid == 0) ? pidx : (lkp ? rank_lookup(*lkp, rank, N - tid * x) : (rank[N - tid * x] & RANK_MASK));
  }
  if (tid == 0) {
    if (block_mode) {
      const uint32_t lc = *lastch;
      if (lc & 0x100u) out[pidx] = (uint8_t)(lc & 0xFFu);  // hole fill: begin[LF[0]] = *end (BWTransform.cpp:60)
    } else {
      out[pidx] = text[pidx];                               // "U[pidx] untouched" (divsufsort.c:506-512)
    }
  }
}

// k_finish_batch — the same per block of a batch (grid = nblocks): block k owns ids and ranks [k*stride, ..+N_k).
// LF[k*256 + j]; nLF_k = nLF for full blocks, nLF_last for the last one (BWTBlock.cpp:104-108 applies per block).
__global__ void __launch_bounds__(256) k_finish_batch(const uint32_t* __restrict__ rank, uint32_t Ntot, uint32_t stride,
                                                      uint32_t nblocks, uint8_t* __restrict__ out,
                                                      uint32_t* __restrict__ LF, uint32_t nLF, uint32_t nLF_last,
                                                      const uint32_t* __restrict__ lastch, LadderState* st,
                                                      const uint32_t* __restrict__ ctrl) {
  const uint32_t k = blockIdx.x, tid = threadIdx.x;
  const uint32_t err = ctrl[CTR_ERR];
  if (k == 0 && tid == 0) st->err = err;
  if (err || st->m != 0u) return;
  const uint32_t start = k * stride;
  const uint32_t Nk = (k + 1u == nblocks) ? Ntot - start : stride;
  const uint32_t nl = (k + 1u == nblocks) ? nLF_last : nLF;
  const uint32_t pidx = (rank[start] & RANK_MASK) - start;
  if (tid < nl) {
    const uint32_t x = Nk / nl;
    LF[k * 256u + tid] = (tid == 0) ? pidx : ((rank[start + Nk - tid * x] & RANK_MASK) - start);
  }
  if (tid == 0) {
    const uint32_t lc = lastch[k];
    if (lc & 0x100u) out[start + pidx] = (uint8_t)(lc & 0xFFu);
  }
}

// =====================================================================================================
// sufcheck on the device (bwtc_cuda_sufcheck, and the verification of bwtc_cuda_divsufsort; DESIGN.md §3.11).
// SA[0..n) is the suffix array of T exactly when
//   (1) it is a permutation of [0, n): every value in range, none twice, and
//   (2) for every r >= 1: (T[SA[r-1]], ISA'[SA[r-1]+1]) < (T[SA[r]], ISA'[SA[r]+1]), ISA' = the inverse of SA with
//       ISA'[n] = -1 standing for the empty suffix
// (neighbours ordered by first byte, then by the rank of their successor, are ordered lexicographically: induction
// on the suffix length).  k_sa_perm scatters ISA[SA[r]] = min r (atomicMin over an all-ones ISA), so a value held twice
// keeps its FIRST row and k_sa_order finds every later one as isa[v] != r.  Failures meet in one 64-bit control word as
// the maximum of ~((phase << 62) | (row << 2) | reason): the host reads the smallest (phase, row) — range and duplicate
// failures (phase 0) before order failures (phase 1, whose ISA is only meaningful for a permutation).
// =====================================================================================================
constexpr int CTR_SA_BAD = 2;  // [2..3] (the words of the inverse's corrupt mask, read back the same way, CTR_INV_BAD)
enum : uint32_t { SA_BAD_RANGE = 1, SA_BAD_DUP = 2, SA_BAD_ORDER = 3 };

__device__ __forceinline__ void sa_fail(uint32_t* ctrl, uint32_t phase, uint32_t row, uint32_t reason) {
  const unsigned long long key = ((unsigned long long)phase << 62) | ((unsigned long long)row << 2) | reason;
  atomicMax(reinterpret_cast<unsigned long long*>(ctrl + CTR_SA_BAD), ~key);
}

// (1a) ranges, and ISA[v] = the first row holding v.  isa[0..n) must hold 0xFFFFFFFF.
__global__ void __launch_bounds__(256) k_sa_perm(const int32_t* __restrict__ sa, uint32_t n, uint32_t* __restrict__ isa,
                                                 uint32_t* __restrict__ ctrl) {
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
    const uint32_t v = (uint32_t)sa[r];  // (a negative value is >= n here)
    if (v >= n) sa_fail(ctrl, 0, r, SA_BAD_RANGE);
    else atomicMin(&isa[v], r);
  }
}

// (1b) duplicates and (2) order.  A warp owns 32 consecutive rows: row r's key (T[SA[r]], ISA'[SA[r]+1] + 1) is
// compared with the key of row r-1, which lane r-1 holds (lane 0 loads it).
__global__ void __launch_bounds__(256) k_sa_order(const uint8_t* __restrict__ text, const int32_t* __restrict__ sa, uint32_t n,
                                                  const uint32_t* __restrict__ isa, uint32_t* __restrict__ ctrl) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  auto key_of = [&](uint32_t v) -> unsigned long long {  // v < n
    const uint32_t succ = (v + 1u < n) ? isa[v + 1u] + 1u : 0u;  // the empty suffix ranks below every other
    return ((unsigned long long)text[v] << 32) | succ;
  };
  for (uint32_t base = warp * 32u; base < n; base += nwarps * 32u) {
    const uint32_t r = base + lane;
    const uint32_t v = (r < n) ? (uint32_t)sa[r] : 0xFFFFFFFFu;
    const bool valid = v < n;
    unsigned long long key = 0;
    if (valid) {
      if (isa[v] != r) sa_fail(ctrl, 0, r, SA_BAD_DUP);
      key = key_of(v);
    }
    unsigned long long pkey = __shfl_up_sync(0xFFFFFFFFu, key, 1);
    bool pvalid = __shfl_up_sync(0xFFFFFFFFu, valid ? 1u : 0u, 1) != 0u;
    if (lane == 0) {
      const uint32_t u = (r > 0u && r < n) ? (uint32_t)sa[r - 1u] : 0xFFFFFFFFu;
      pvalid = u < n;
      pkey = pvalid ? key_of(u) : 0ull;
    }
    if (valid && pvalid && r > 0u && !(pkey < key)) sa_fail(ctrl, 1, r, SA_BAD_ORDER);
  }
}

// Test hook (BWTC_DEBUG_CORRUPT_SA=r): swap SA[r] and SA[r+1] before the verification checks them.
__global__ void k_debug_swap_sa(int32_t* sa, uint32_t r) {
  const int32_t a = sa[r];
  sa[r] = sa[r + 1u];
  sa[r + 1u] = a;
}

}  // namespace bwtc_b200
