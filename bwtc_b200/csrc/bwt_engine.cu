// bwtc_b200/csrc/bwt_engine.cu — host orchestration + extern "C" layer (include/bwtc_cuda.h) of the
// B200-native forward-BWT engine.  Host code is C++; all compute is in bwt_kernels.cuh.
// No CPU fallback anywhere: if the device, an allocation or a kernel fails the call returns a negative
// code and bwtc_cuda_last_error() says why.
#include "../../include/bwtc_cuda.h"
#include "bwt_kernels.cuh"
#include "ibwt_kernels.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

using namespace bwtc_b200;

namespace {

constexpr int RS_BLOCK = BWTC_RS_BLOCK;
constexpr int RS_IPT64 = BWTC_RS_IPT64;
constexpr int RS_IPT32 = BWTC_RS_IPT32;
constexpr uint32_t RS_TILE64 = RS_BLOCK * RS_IPT64;
constexpr uint32_t RS_TILE32 = RS_BLOCK * RS_IPT32;
constexpr uint32_t AUX_TILE = 2048;  // k_pack_round0 / k_build_keys / k_rerank tile
constexpr int MAX_PASSES = 8;
constexpr uint32_t GRAM_OFF = MAX_PASSES * 512;    // the gram histogram of k_pack_round0 sits behind the digit histograms
constexpr uint32_t HIST_WORDS = GRAM_OFF + (1u << GRAM_BITS);  // digit histograms of one sort: pass p at p << rb (rb = 8 or 9 bits)
// Words per look-back status row: 256 (8-bit digits), 512 when the 9-bit digit passes are enabled (BWTC_RADIX9=1).
inline uint32_t status_row_words_for(int use_radix9) { return use_radix9 ? 512u : 256u; }
inline int env_radix9() { const char* e = getenv("BWTC_RADIX9"); return e ? atoi(e) : 0; }
constexpr uint32_t TEXT_PAD = 64;

thread_local char g_err[512] = "";

void set_err(char* dst, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(dst, 512, fmt, ap);
  va_end(ap);
}

inline uint32_t ceil_log2_u64(uint64_t v) {  // smallest b with 2^b >= v  (v >= 1)
  uint32_t b = 0;
  while ((1ull << b) < v) ++b;
  return b;
}
inline uint32_t div_up(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }

}  // namespace

constexpr uint32_t MAX_BATCH = BWTC_CUDA_MAX_BATCH;  // blocks sorted as one text (6 key bits for the block number)
constexpr uint32_t LF_PARK = MAX_BATCH * 256, LF_WORDS = LF_PARK + MAX_BATCH + 8;
// Pinned staging ring for PAGEABLE caller buffers (a malloc'ed PrecompressorBlock, PrecompressorBlock.cpp:37-49): the
// worker thread copies chunk by chunk through it while the DMA engine moves the previous chunks, on copy streams of
// their own.  Pinned caller buffers are copied directly.
constexpr size_t RING_CHUNK = 4u << 20;
constexpr int RING_SLOTS = 4;
constexpr uint32_t KTAB_BITS = 20;  // lazy ranks: prefix table of the sorted round-0 keys (4 MiB)

struct bwtc_cuda_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;     // kernels (+ the direct copies of pinned / device-resident caller buffers)
  cudaStream_t s_in = nullptr, s_out = nullptr;  // staged H2D / D2H of pageable caller buffers (pinned ring)
  cudaEvent_t ev_sync = nullptr;     // host waits (blocking-sync event unless spin_wait)
  cudaEvent_t ev_in = nullptr, ev_comp = nullptr;  // hand-off copy stream <-> kernel stream
  cudaEvent_t ev_ring[RING_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
  uint8_t* h_ring = nullptr;         // RING_SLOTS x RING_CHUNK pinned bytes, allocated on first use
  uint64_t ring_next = 0;            // slots are handed out round-robin across calls ...
  bool ring_busy[RING_SLOTS] = {false, false, false, false};  // ... and waited for (ev_ring) before they are reused
  int poll_spin_us = 150, poll_sleep_us = 40;
  int wait_mode = 0;                 // host waits: 0 adaptive (poll briefly, then sleep in short steps), 1 spin
                                     // (cudaStreamSynchronize), 2 blocking-sync event
  uint32_t cap = 0;  // max block bytes (a batch: sum of block bytes + blocks - 1)
  size_t max_rs_tiles = 0, max_aux_tiles = 0;
  // ---- device memory (DESIGN.md §3.1)
  uint8_t* d_in = nullptr;        // staged input block(s); scratch once the text exists
  uint8_t* d_text = nullptr;      // T' = reverse(X) . 0x00 (+ padding)
  uint8_t* d_out = nullptr;       // BWT bytes by rank
  uint32_t* d_rank = nullptr;     // inverse suffix array, bit 31 = final
  void* d_keys[2] = {nullptr, nullptr};      // ping-pong sort keys (8N bytes each); between sorts: 2 x 2 u32[N] work arrays
  uint32_t* d_idx[2] = {nullptr, nullptr};   // ping-pong suffix ids; between sorts: 2 u32[N] work arrays
  uint8_t* d_aux[2] = {nullptr, nullptr};    // ping-pong one-byte payload of the round-0 sort (predecessor codes), N each
  uint32_t* d_scat = nullptr;     // u32[N]: staged ranks of the bucketed scatter (the ids go to the idle id buffer)
  uint32_t* d_zero = nullptr;     // [ctrl CTR_WORDS][hist HIST_WORDS][tstate rows of max_aux_tiles] zeroed per round
  uint32_t* d_status = nullptr;   // [MAX_PASSES][LB_PAD_ROWS + max_rs_tiles][status_row_words] radix look-back words; the pad rows in
                                  // front of every pass hold "prefix 0" for ever, so a walk needs no bounds check
  uint32_t* d_tilecnt = nullptr;  // [2][max_aux_tiles]: per-tile live counts of k_rerank and their exclusive prefix,
                                  // then [max_aux_tiles][MAX_RERANK_WINDOWS+1] bucket offsets of the bucketed scatter
  uint32_t* d_LF = nullptr;       // [LF_PARK) LFpowers (one row of 256 per block of a batch), [LF_PARK + k] parked hole byte
                                  // of block k
  uint32_t* d_livebits = nullptr; // lazy ranks: bit i = rank[i] is stored (N / 32 words)
  uint32_t* d_ktab = nullptr;     // lazy ranks: first sorted position per key prefix ((1 << KTAB_BITS) + 2 words)
  LookupParams* d_lookup = nullptr;  // ... what rank_lookup needs, in device memory
  LookupParams* h_lookup = nullptr;  // (pinned host copy)
  LadderState* d_state = nullptr; // device-side round control (bwt_kernels.cuh)
  LadderState* h_state = nullptr; // ... its pinned host copy
  unsigned long long* d_wtab = nullptr;  // window-sample table: WS_SLOTS keys, WS_SLOTS counters, 2 doubles
  uint32_t* d_bhist = nullptr;    // [MAX_BATCH][256] per-block byte histograms of a batch
  const uint8_t** d_bptr = nullptr;  // [MAX_BATCH] device pointers to the blocks of a batch
  int32_t* d_sa = nullptr;        // suffix array of bwtc_cuda_divsufsort (host variant): 4 (cap + 1) bytes, allocated by its
                                  // first call, not counted by bwtc_cuda_scratch_bytes
  // ---- pinned host memory
  uint32_t* h_small = nullptr;    // [ctrl CTR_WORDS][hist HIST_WORDS][LF 256 + pair statistics]
  uint8_t* h_batch = nullptr;     // [MAX_BATCH] pointers, [MAX_BATCH][256] histograms, [MAX_BATCH][256] LFpowers
  // ---- timing
  cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
  std::vector<cudaEvent_t> ev_pool;
  int timing_detail = 0;
  // ---- policy knobs (defaults are the measured optimum on B200; the environment variables in bwtc_cuda_ctx_create
  //      exist so that tests can force every code path, see tests/test_gpu_parity.py)
  int static_tiles = 1;           // look-back kernels take blockIdx.x as tile id (0: dynamic tickets); cleared for good
                                  // if the spin watchdog ever fires
  int lb_watchdog = 0;            // the last transform failed on the look-back watchdog
  int debug_fake_watchdog = 0;    // test hook: pretend the watchdog fired while static tile ids are in use
  int debug_reverse_tiles = 0;    // test hook: static tile ids in REVERSE dispatch order (a real violation)
  int verify = 0;                 // forward outputs are inverted on the device and compared (DESIGN.md §3.10); BWTC_VERIFY
  int debug_corrupt_out = 0;      // test hook: one byte of the forward output is changed before it is verified
  uint32_t debug_corrupt_lf = 0;  // test hook (j >= 1): LFpowers[j] is changed on the device before it is verified
  int64_t debug_corrupt_sa = -1;  // test hook (r >= 0): SA[r] and SA[r+1] are swapped on the device before they are verified
  int d2h_kernel = 0;             // BWTC_D2H_KERNEL=1: result copies to pinned host buffers by a copying kernel (k_copy_out)
                                  // instead of the copy engine — measured no better (profiles/r02_experiments.md), kept as a knob
  int d2h_ctas = 16;
  int debug_skip_copies = 0;      // timing experiments only (bit 0: no H2D of host blocks, bit 1: no D2H): results are WRONG
  int ladder_first = 2, ladder_more = 4;  // segmented rounds enqueued speculatively behind a sort round / per retry
  int use_radix9 = 0;             // BWTC_RADIX9=1: 9-bit digits for 64-bit-key sorts whenever that saves a pass.  Measured
                                  // slower (a 9-bit pass costs +23%, 7 of them more than 8 eight-bit ones): kept as an
                                  // experiment, profiles/r02_experiments.md
  uint32_t status_row_words = 256;
  int use_partial = 1;            // spare low bits of the round-0 key take the top bits of the next character (BWTC_PARTIAL=0: zeros)
  int use_gram = 1;               // round-0 digit histograms projected from one 12-bit gram histogram (6- and 3-bit codes; BWTC_GRAM=0:
                                  // counted per digit class + k_hist_derive)
  int twopass = 0;                // BWTC_TWOPASS=1: with two L2 windows the second window is scattered by k_scatter_window from the
                                  // rank words the first k_rerank launch stored in sorted order, instead of a second k_rerank
                                  // launch (measured: Markov 32 MiB equal, source text -3%; the random scatter itself is the cost)
  int hybrid2 = 0;                // BWTC_HYBRID2=1: with two L2 windows, window 0 is written directly and window 1 staged + one
                                  // k_scatter_bucket, instead of one k_rerank launch per window (measured equal: 2.90 vs 2.88 ms)
  uint32_t rerank_pf_tiles = 0;   // k_rerank: L2 prefetch distance in tiles (BWTC_RERANK_PF; 0 = off)
  int use_lazy = 1;               // lazy ranks after round 0 (DESIGN.md §3.9): 0 never, 1 when the key-shape policy predicts
                                  // that few suffixes stay in groups, 2 always (tests)
  uint32_t lazy_min_suffixes = 4u << 20;
  double lazy_max_live = 0.09;    // i.i.d.-like blocks: at most this predicted live fraction after round 0.  Measured with the
                                  // look-up-free segmented rounds: random bytes 256 / 384 MiB (6.1% / 8.9%) -8% / -5%
  double lazy_max_repeats = 32.0; // blocks with memory: at most this many other positions share a position's 8-gram (Markov
                                  // 16 / 32 / 64 MiB: 1.3 / 3.0 / 5.2; repetitive 16 MiB: ~3800, source text ~1.5e5)
  int use_seg = 1;                // segmented (sort-free) doubling rounds when every group is small
  int use_batch = 1;              // small equal-sized blocks of one call are sorted as one text
  int use_pack_pred = 1;          // carry code(T[id-1]) above the id through the round-0 sort when it fits
  uint32_t aux_min_suffixes = 96u << 20;  // ... else, from this many suffixes on, as a one-byte payload array (0 = never)
  int bucket_min_windows = 3;     // bucketed rank scatter from this many L2 windows on (0 = never)
  uint64_t rerank_window_bytes = 72ull << 20;  // rank-scatter window kept L2-resident (126 MB L2)
  uint32_t force_chars = 0, force_keybytes = 0;
  uint32_t debug_max_rounds = 0;  // != 0: stop refining after this many rounds (results are then wrong on purpose)
  int last_cur = 0;               // sort buffer holding the last round's sorted records
  RerankParams rr0;               // round-0 re-rank parameters of the block in flight (fallback out of lazy ranks)
  bwtc_cuda_stats stats;
  char err[512];
  uint32_t* d_ctrl() const { return d_zero; }
  uint32_t* d_hist() const { return d_zero + CTR_WORDS; }
  unsigned long long* d_tstate() const { return reinterpret_cast<unsigned long long*>(d_zero + CTR_WORDS + HIST_WORDS); }
  uint32_t* h_ctrl() const { return h_small; }
  uint32_t* h_hist() const { return h_small + CTR_WORDS; }
  uint32_t* h_LF() const { return h_small + CTR_WORDS + HIST_WORDS; }
};

#define CK(ctx, call)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      set_err((ctx)->err, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, __LINE__,  \
              cudaGetErrorString(e_));                                                             \
      return BWTC_CUDA_ECUDA;                                                                      \
    }                                                                                              \
  } while (0)

namespace {

template <typename KeyT, int IPT, bool IOTA, bool AUX, int RB = 8>
int set_pass_attr(bwtc_cuda_ctx* ctx) {
  CK(ctx, cudaFuncSetAttribute(k_radix_pass<KeyT, RS_BLOCK, IPT, IOTA, AUX, RB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)RadixPassSmem<KeyT, RS_BLOCK, IPT, AUX, RB>::bytes));
  return 0;
}

void ctx_free(bwtc_cuda_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  cudaFree(c->d_in); cudaFree(c->d_text); cudaFree(c->d_out); cudaFree(c->d_rank);
  cudaFree(c->d_keys[0]); cudaFree(c->d_keys[1]); cudaFree(c->d_idx[0]); cudaFree(c->d_idx[1]);
  cudaFree(c->d_zero); cudaFree(c->d_status); cudaFree(c->d_LF); cudaFree(c->d_wtab); cudaFree(c->d_tilecnt); cudaFree(c->d_scat);
  cudaFree(c->d_bhist); cudaFree(c->d_bptr); cudaFree(c->d_aux[0]); cudaFree(c->d_aux[1]);
  cudaFree(c->d_state); cudaFree(c->d_livebits); cudaFree(c->d_ktab); cudaFree(c->d_lookup); cudaFree(c->d_sa);
  if (c->h_lookup) cudaFreeHost(c->h_lookup);
  if (c->h_batch) cudaFreeHost(c->h_batch);
  if (c->h_small) cudaFreeHost(c->h_small);
  if (c->h_state) cudaFreeHost(c->h_state);
  if (c->h_ring) cudaFreeHost(c->h_ring);
  if (c->ev_begin) cudaEventDestroy(c->ev_begin);
  if (c->ev_end) cudaEventDestroy(c->ev_end);
  if (c->ev_sync) cudaEventDestroy(c->ev_sync);
  if (c->ev_in) cudaEventDestroy(c->ev_in);
  if (c->ev_comp) cudaEventDestroy(c->ev_comp);
  for (cudaEvent_t e : c->ev_ring) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
  if (c->s_in) cudaStreamDestroy(c->s_in);
  if (c->s_out) cudaStreamDestroy(c->s_out);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

struct Round0Plan {
  uint32_t sigma, bits, chars, keybytes, npass;
  uint32_t rb;        // digit width of the round-0 sort: 9 when that saves a pass over 8-bit digits (64-bit keys only)
  uint32_t rbits;     // spare low key bits filled with the top bits of character c+1 (PackParams::rbits)
  PackParams pp;
  bool has_memory;    // the 8-gram sample says the source is not i.i.d.-like (text, repeats)
  double live_pred;   // i.i.d.-like sources: predicted fraction of suffixes still tied after round 0, L(chars)
  double repeats;     // mean number of other text positions sharing a position's 8-gram (N x sampled pair collision rate)
};

// Dense alphabet + round-0 key shape (DESIGN.md §3.2).  present[c] != 0 for every byte of the text.
// blk_bits > 0 (batch of blocks sorted as one text): code 0 is reserved for the sentinel positions, and blk_bits key
// bits above the characters hold the block number.
void plan_round0(const bwtc_cuda_ctx* ctx, const uint64_t* count, const bool* present, uint32_t N,
                 const double* pair_stats, Round0Plan* pl, uint32_t blk_bits = 0) {
  uint32_t sigma = blk_bits ? 1u : 0u;
  double total = 0, H0 = 0;
  for (int c = 0; c < 256; ++c) {
    pl->pp.lut[c] = 0;
    if (present[c]) { pl->pp.lut[c] = (uint8_t)sigma; ++sigma; total += (double)count[c]; }
  }
  if (sigma > 256) sigma = 256;  // 256 data bytes + reserved sentinel: handled by the caller (falls back to single blocks)
  for (int c = 0; c < 256; ++c)
    if (present[c] && count[c]) { double p = (double)count[c] / total; H0 -= p * std::log2(p); }
  const uint32_t b = sigma <= 2 ? 1 : ceil_log2_u64(sigma);
  const uint32_t cmax64 = (64 - blk_bits) / b, cmax32 = blk_bits >= 32 - b ? 0u : (32 - blk_bits) / b;
  uint32_t chars, keybytes;
  if (ctx->force_chars || ctx->force_keybytes) {
    keybytes = (ctx->force_keybytes == 4 && cmax32 >= 1) ? 4 : 8;
    const uint32_t cmax = keybytes == 4 ? cmax32 : cmax64;
    chars = ctx->force_chars ? ctx->force_chars : cmax;
    if (chars > cmax) chars = cmax;
    if (chars < 1) chars = 1;
  } else {
    // Does the source have memory?  Compare the MEASURED collision rate of sampled 8-byte windows with the rate
    // an i.i.d. source with this byte histogram would show, (sum q^2)^8.  Text and repeats exceed it by orders
    // of magnitude: they keep many suffixes tied whatever the order-0 statistics say, and every extra character
    // ordered in round 0 is far cheaper than a doubling round over the suffixes it would leave live (measured:
    // profiles/r01_experiments.md), so their 64-bit key is filled completely.
    double q2 = 0.0;
    for (int c = 0; c < 256; ++c)
      if (present[c] && count[c]) { const double q = (double)count[c] / total; q2 += q * q; }
    const double samples = pair_stats[1];
    const double all_pairs = samples * (samples - 1.0) * 0.5;
    const double expected = all_pairs * std::pow(q2, 8.0);
    const bool has_memory = (H0 < 1e-3) || samples < 64.0 || (pair_stats[0] > 8.0 * expected + 16.0);
    if (has_memory) {
      keybytes = 8;
      chars = cmax64;
    } else {
      // i.i.d.-like source (random bytes, DNA): a suffix stays tied after c characters with probability
      // L(c) = 1 - exp(-N 2^(-H0 c)).  One digit pass over a record costs about the same for 8- and 12-byte
      // records (the pass is latency-, not byte-bound), a doubling round costs ~npd+2 pass-equivalents per
      // live record: pick the c that minimises  ceil(c b / 8) + L(c) (npd + 2).
      const double npd = std::ceil((2.0 * std::log2((double)N + 2.0)) / 8.0);
      double best = 1e300;
      chars = cmax64;
      for (uint32_t c = 1; c <= cmax64; ++c) {
        const double p0 = std::ceil(((double)c * b + blk_bits) / 8.0) * ((uint64_t)c * b + blk_bits > 32 ? 1.1 : 1.0);
        const double L = 1.0 - std::exp(-(double)N * std::exp2(-H0 * (double)c));
        const double cost = p0 + L * (npd + 2.0);
        if (cost < best - 1e-9) { best = cost; chars = c; }
      }
      // use every bit of the last digit pass that is executed anyway
      const uint32_t np = div_up((uint64_t)chars * b + blk_bits, 8);
      const uint32_t cfull = (8 * np - blk_bits) / b;
      const uint32_t cap = ((uint64_t)chars * b + blk_bits <= 32) ? cmax32 : cmax64;
      chars = cfull < cap ? cfull : cap;
      keybytes = ((uint64_t)chars * b + blk_bits <= 32) ? 4 : 8;
    }
  }
  pl->has_memory = true;
  pl->live_pred = 1.0;
  pl->repeats = HUGE_VAL;
  if (!(ctx->force_chars || ctx->force_keybytes)) {
    double q2 = 0.0;
    for (int c = 0; c < 256; ++c)
      if (present[c] && count[c]) { const double q = (double)count[c] / total; q2 += q * q; }
    const double samples = pair_stats[1];
    const double all_pairs = samples * (samples - 1.0) * 0.5;
    const double expected = all_pairs * std::pow(q2, 8.0);
    pl->has_memory = (H0 < 1e-3) || samples < 64.0 || (pair_stats[0] > 8.0 * expected + 16.0);
    if (!pl->has_memory) pl->live_pred = 1.0 - std::exp(-(double)N * std::exp2(-H0 * (double)chars));
    if (samples >= 64.0) pl->repeats = pair_stats[0] / all_pairs * (double)N;
  }
  pl->sigma = sigma;
  pl->bits = b;
  pl->chars = chars;
  pl->keybytes = keybytes;
  pl->npass = div_up((uint64_t)chars * b + blk_bits, 8);
  pl->rb = 8;
  if (ctx->use_radix9 && keybytes == 8 && div_up((uint64_t)chars * b + blk_bits, 9) < pl->npass) {
    pl->rb = 9;
    pl->npass = div_up((uint64_t)chars * b + blk_bits, 9);
  }
  {
    // the digit passes cover rb * npass bits (at most the key width): what the c characters leave over takes the top bits
    // of the next character (never a whole one: the chooser above already uses every whole character that fits)
    const uint32_t covered = std::min<uint32_t>(pl->rb * pl->npass, keybytes * 8u);
    const uint32_t used = chars * b + blk_bits;
    uint32_t r = (ctx->use_partial && blk_bits == 0 && covered > used) ? covered - used : 0u;
    if (r >= b) r = b - 1u;
    if (chars >= 64u) r = 0;
    pl->rbits = r;
  }
  pl->pp.rbits = pl->rbits;
  pl->pp.bits = b;
  pl->pp.chars = chars;
  pl->pp.nblocks = 1;
  pl->pp.stride = 0;
}

// Number of id windows the rank scatter of a round is split into (k_rerank RerankParams::win_lo/hi).
uint32_t rerank_windows(const bwtc_cuda_ctx* ctx, uint32_t N, uint32_t m) {
  if ((uint64_t)m * 4 < (uint64_t)N) return 1;  // few scattered writes: a second read of the records costs more
  uint64_t w = ((uint64_t)N * 4 + ctx->rerank_window_bytes - 1) / ctx->rerank_window_bytes;
  if (w < 1) w = 1;
  if (!ctx->bucket_min_windows && w > 8) w = 8;  // per-window re-reads: beyond 8 they cost more than the L2 residency saves
  if (w > MAX_RERANK_WINDOWS) w = MAX_RERANK_WINDOWS;
  return (uint32_t)w;
}

// Number of k_rerank launches (= look-back word rows to zero): one in bucket mode, else one per window.
uint32_t rerank_launches(const bwtc_cuda_ctx* ctx, uint32_t N, uint32_t m) {
  const uint32_t w = rerank_windows(ctx, N, m);
  return (ctx->bucket_min_windows && w >= (uint32_t)ctx->bucket_min_windows) ? 1u : w;
}

inline bool dbg_any(const bwtc_cuda_ctx* ctx) { return ctx->debug_max_rounds != 0; }

// Tile-id source of the look-back kernels: the block index (default), tickets, or the reversed debug map.
inline uint32_t tile_slot(const bwtc_cuda_ctx* ctx, uint32_t ticket_word) {
  if (!ctx->static_tiles) return ticket_word;
  return ctx->debug_reverse_tiles ? CTR_STATIC_REV : CTR_STATIC;
}

// Row 0 of the look-back status words of digit pass p (LB_PAD_ROWS rows of "prefix 0" words sit in front of it, for
// either row width).
inline uint32_t* status_rows(const bwtc_cuda_ctx* ctx, int p) {
  return ctx->d_status + ((size_t)p * (ctx->max_rs_tiles + LB_PAD_ROWS) + LB_PAD_ROWS) * ctx->status_row_words;
}

struct PassTimer {
  bwtc_cuda_ctx* ctx;
  size_t used = 0;
  int begin() {
    if (!ctx->timing_detail) return 0;
    if (used + 2 > ctx->ev_pool.size()) return 0;
    CK(ctx, cudaEventRecord(ctx->ev_pool[used], ctx->stream));
    return 0;
  }
  int end() {
    if (!ctx->timing_detail) return 0;
    if (used + 2 > ctx->ev_pool.size()) return 0;
    CK(ctx, cudaEventRecord(ctx->ev_pool[used + 1], ctx->stream));
    used += 2;
    return 0;
  }
};

// One LSD radix sort of m records: executes the digit passes whose bit is set in pass_mask, ping-ponging
// between buffer 0 and 1.  Records start in buffer `cur` (0); returns the buffer holding the result.
template <typename KeyT, int IPT, bool AUX, int RB = 8>
int run_sort_impl(bwtc_cuda_ctx* ctx, uint32_t m, uint32_t pass_mask, bool first_iota, uint32_t iota_top, int* cur_io,
                  PassTimer* pt, uint32_t* passes_done, uint32_t pack_bits, uint32_t topshift, uint32_t pred_mask) {
  constexpr uint32_t TILE = RS_BLOCK * IPT;
  const uint32_t tiles = div_up(m, TILE);
  const size_t smem = RadixPassSmem<KeyT, RS_BLOCK, IPT, AUX, RB>::bytes;
  int cur = *cur_io;
  bool iota = first_iota;
  uint32_t done = 0;
  for (int p = 0; p < MAX_PASSES; ++p) {
    if (!((pass_mask >> p) & 1u)) continue;
    const KeyT* kin = static_cast<const KeyT*>(ctx->d_keys[cur]);
    KeyT* kout = static_cast<KeyT*>(ctx->d_keys[cur ^ 1]);
    uint32_t* status = status_rows(ctx, p);
    if (pt->begin()) return BWTC_CUDA_ECUDA;
    if (iota)
      k_radix_pass<KeyT, RS_BLOCK, IPT, true, AUX, RB><<<tiles, RS_BLOCK, smem, ctx->stream>>>(
          kin, nullptr, kout, ctx->d_idx[cur ^ 1], m, (uint32_t)RB * p, ctx->d_hist() + ((size_t)p << RB), status, ctx->d_ctrl(),
          tile_slot(ctx, (uint32_t)(CTR_PASS0 + p)), iota_top, pack_bits, topshift, pred_mask, nullptr,
          ctx->d_aux[cur ^ 1]);
    else
      k_radix_pass<KeyT, RS_BLOCK, IPT, false, AUX, RB><<<tiles, RS_BLOCK, smem, ctx->stream>>>(
          kin, ctx->d_idx[cur], kout, ctx->d_idx[cur ^ 1], m, (uint32_t)RB * p, ctx->d_hist() + ((size_t)p << RB), status,
          ctx->d_ctrl(), tile_slot(ctx, (uint32_t)(CTR_PASS0 + p)), iota_top, 0u, 0u, 0u, ctx->d_aux[cur], ctx->d_aux[cur ^ 1]);
    CK(ctx, cudaGetLastError());
    if (pt->end()) return BWTC_CUDA_ECUDA;
    ctx->stats.kernel_launches++;
    const uint64_t rec = sizeof(KeyT) + 4 + (AUX ? 1 : 0);
    ctx->stats.algorithmic_bytes += (uint64_t)m * (2 * rec - (iota ? 4 + (AUX ? 1 : 0) : 0));
    ctx->stats.sort_bytes += (uint64_t)m * (2 * rec - (iota ? 4 + (AUX ? 1 : 0) : 0));
    ctx->stats.sort_launches++;
    iota = false;
    cur ^= 1;
    ++done;
  }
  *cur_io = cur;
  *passes_done = done;
  return 0;
}

// One LSD radix sort of m records: executes the digit passes whose bit is set in pass_mask, ping-ponging
// between buffer 0 and 1.  Records start in buffer `cur` (0); returns the buffer holding the result.
// aux: a one-byte payload (predecessor character code) is produced by the first pass and carried along.
// rb: digit width, 8 or 9 bits (9 only for 64-bit keys); pass p sorts on bits [rb*p, rb*p + rb).
template <typename KeyT, int IPT>
int run_sort(bwtc_cuda_ctx* ctx, uint32_t m, uint32_t pass_mask, bool first_iota, uint32_t iota_top, int* cur_io,
             PassTimer* pt, uint32_t* passes_done, uint32_t pack_bits = 0, uint32_t topshift = 0,
             uint32_t pred_mask = 0xFFFFFFFFu, bool aux = false, uint32_t rb = 8) {
  if constexpr (sizeof(KeyT) == 8) {
    if (rb == 9) {
      if (aux)
        return run_sort_impl<KeyT, IPT, true, 9>(ctx, m, pass_mask, first_iota, iota_top, cur_io, pt, passes_done, pack_bits,
                                                 topshift, pred_mask);
      return run_sort_impl<KeyT, IPT, false, 9>(ctx, m, pass_mask, first_iota, iota_top, cur_io, pt, passes_done, pack_bits,
                                                topshift, pred_mask);
    }
  }
  if (rb != 8) { set_err(ctx->err, "run_sort: %u-bit digits are not built for this key type", rb); return BWTC_CUDA_EINTERNAL; }
  if (aux)
    return run_sort_impl<KeyT, IPT, true>(ctx, m, pass_mask, first_iota, iota_top, cur_io, pt, passes_done, pack_bits, topshift,
                                          pred_mask);
  return run_sort_impl<KeyT, IPT, false>(ctx, m, pass_mask, first_iota, iota_top, cur_io, pt, passes_done, pack_bits, topshift,
                                         pred_mask);
}

int zero_round_state(bwtc_cuda_ctx* ctx, uint32_t N, uint32_t m, uint32_t rs_tile, uint32_t pass_mask, uint32_t rb = 8) {
  const uint32_t aux_tiles = div_up(m, AUX_TILE);
  CK(ctx, cudaMemsetAsync(ctx->d_zero + CTR_STICKY, 0,
                          (size_t)(CTR_WORDS - CTR_STICKY + HIST_WORDS) * 4 + (size_t)rerank_launches(ctx, N, m) * ctx->max_aux_tiles * 8,
                          ctx->stream));
  const uint32_t tiles = div_up(m, rs_tile);
  for (int p = 0; p < MAX_PASSES; ++p)
    if ((pass_mask >> p) & 1u)
      CK(ctx, cudaMemsetAsync(status_rows(ctx, p), 0, ((size_t)tiles * 4u) << rb, ctx->stream));
  return 0;
}

// k_rerank over the m sorted records in buffer `cur`, plus the rank scatter.  A rank[] array that needs three or
// more L2 windows is written bucket by bucket (ONE k_rerank launch stages (id, rank) pairs per id bucket, one
// k_scatter_bucket launch per bucket reads them back); with two windows re-running k_rerank per window is
// as fast (measured) and needs no staging.
template <typename KeyT, bool ROUND0>
int launch_rerank(bwtc_cuda_ctx* ctx, int cur, uint32_t m, uint32_t N, RerankParams rp, const EmitParams& ep,
                  uint32_t* stage_nr, uint32_t* stage_id, bool single_window = false, bool no_stage = false) {
  cudaStream_t st = ctx->stream;
  const uint32_t tiles = div_up(m, AUX_TILE);
  const uint32_t nwin = single_window ? 1u : rerank_windows(ctx, N, m);
  const KeyT* keys = static_cast<const KeyT*>(ctx->d_keys[cur]);
  uint32_t* woff = ctx->d_tilecnt + 2 * ctx->max_aux_tiles;
  // (ep.sa: the instantiation that also writes the suffix array)
  auto rerank = [&](unsigned long long* tstate, const StageParams& sp) {
    if (ROUND0 && rp.lazy) {
      if (ep.sa) k_rerank<KeyT, ROUND0, ROUND0, true><<<tiles, 256, 0, st>>>(keys, ctx->d_idx[cur], ctx->d_rank, rp, tstate, ctx->d_ctrl(), ep, sp);
      else k_rerank<KeyT, ROUND0, ROUND0><<<tiles, 256, 0, st>>>(keys, ctx->d_idx[cur], ctx->d_rank, rp, tstate, ctx->d_ctrl(), ep, sp);
    } else {
      if (ep.sa) k_rerank<KeyT, ROUND0, false, true><<<tiles, 256, 0, st>>>(keys, ctx->d_idx[cur], ctx->d_rank, rp, tstate, ctx->d_ctrl(), ep, sp);
      else k_rerank<KeyT, ROUND0><<<tiles, 256, 0, st>>>(keys, ctx->d_idx[cur], ctx->d_rank, rp, tstate, ctx->d_ctrl(), ep, sp);
    }
  };
  const bool hybrid2 = ctx->hybrid2 && nwin == 2u && !(ROUND0 && rp.lazy);
  if ((ctx->bucket_min_windows && nwin >= (uint32_t)ctx->bucket_min_windows) || hybrid2) {
    const uint32_t win_ids = div_up(N, nwin);
    rp.win_lo = 0;
    rp.win_hi = 0xFFFFFFFFu;
    rp.emit = 1;
    rp.pf_tiles = ctx->rerank_pf_tiles;
    rp.ctr_slot = tile_slot(ctx, (uint32_t)CTR_RERANK);
    rp.nbuckets = nwin;
    rp.nr_out = nullptr;
    rp.direct0 = hybrid2 ? 1u : 0u;
    rp.bucket_magic = (uint32_t)(((1ull << 32) + win_ids - 1) / win_ids);
    StageParams sp{stage_nr, stage_id, ctx->d_tilecnt, no_stage ? 0 : 1, ctx->d_idx[cur ^ 1], ctx->d_scat, woff};
    rerank(ctx->d_tstate(), sp);
    const uint32_t grid = std::min<uint32_t>(div_up(tiles, 8), (uint32_t)ctx->sm_count * 8u);
    for (uint32_t b = hybrid2 ? 1u : 0u; b < nwin; ++b)
      k_scatter_bucket<<<grid, 256, 0, st>>>(ctx->d_idx[cur ^ 1], ctx->d_scat, woff, tiles, nwin, b, AUX_TILE, ctx->d_rank, ctx->d_ctrl());
    CK(ctx, cudaGetLastError());
    ctx->stats.kernel_launches += 1 + nwin - (hybrid2 ? 1u : 0u);
    ctx->stats.algorithmic_bytes += (uint64_t)m * (hybrid2 ? 8 : 16);  // staged (id, rank) pairs: written once, read once
    return 0;
  }
  // Two windows: the first launch also leaves every record's new rank word beside its id (d_scat, idle here), and the
  // second window is served by the light k_scatter_window instead of a second full re-rank.
  const bool twopass = ctx->twopass && nwin == 2u && !(ROUND0 && rp.lazy);
  for (uint32_t w = 0; w < nwin; ++w) {
    rp.win_lo = (uint32_t)((uint64_t)N * w / nwin);
    rp.win_hi = (w + 1 == nwin) ? 0xFFFFFFFFu : (uint32_t)((uint64_t)N * (w + 1) / nwin);
    rp.nr_out = (twopass && w == 0) ? ctx->d_scat : nullptr;
    if (twopass && w == 1) {
      const uint32_t grid = std::min<uint32_t>(div_up(m, 1024u), (uint32_t)ctx->sm_count * 8u);
      const uint32_t mask = ROUND0 ? rp.id_mask : 0x7FFFFFFFu;
      k_scatter_window<<<grid, 256, 0, st>>>(ctx->d_idx[cur], ctx->d_scat, m, mask, rp.win_lo, rp.win_hi, ctx->d_rank, ctx->d_ctrl());
      CK(ctx, cudaGetLastError());
      ctx->stats.kernel_launches++;
      ctx->stats.algorithmic_bytes += (uint64_t)m * 12;  // rank words written once, ids + rank words read once
      break;
    }
    // round 0: the first window launch emits every BWT byte (whole words); so does the only k_rerank launch of a two-pass
    // scatter in any round; otherwise every window launch emits for its own ids
    rp.emit = (ROUND0 || twopass) ? (w == 0 ? 1u : 2u) : 0u;
    rp.pf_tiles = ctx->rerank_pf_tiles;
    rp.ctr_slot = tile_slot(ctx, (uint32_t)(CTR_RERANK + w));
    rp.nbuckets = 0;
    rp.direct0 = 0;
    rp.bucket_magic = 0;
    StageParams sp{stage_nr, stage_id, ctx->d_tilecnt, (w == 0 && !no_stage) ? 1 : 0, nullptr, nullptr, nullptr};
    rerank(ctx->d_tstate() + (size_t)w * ctx->max_aux_tiles, sp);
    CK(ctx, cudaGetLastError());
    ctx->stats.kernel_launches++;
  }
  return 0;
}

// A batch of small blocks transformed as ONE suffix-sorting problem (DESIGN.md §3.6): text = T'_0 T'_1 ... with
// T'_k = reverse(X_k) . 0x00 at offset k * (n0 + 1).  All blocks have n0 bytes, the last one n_last <= n0.
struct BatchSpec {
  uint32_t nblocks, n0, n_last;
  const void* const* in;  // per block: host pointers, or device pointers when on_device
  void* const* out;
  bool on_device;
  uint32_t* LF;           // [nblocks][256]
  uint32_t nLF, nLF_last; // LFpowers per full block / for the last block
  uint32_t* freqs;        // [nblocks][256] incremented, or nullptr
};
constexpr int64_t BATCH_NEEDS_SINGLE = -1000;  // all 256 byte values present: no code left for the reserved sentinel

// One transform call: what the caller handed in, and what phase A (input + policy) learnt about it.
struct Job {
  bool block_mode = true;          // in = X (n block bytes), result n bytes;  false (raw): in = T (n bytes)
  const uint8_t* h_in = nullptr;   // host buffers of a single block ...
  uint8_t* h_out = nullptr;
  const uint8_t* in_dev = nullptr; // ... or the caller's device buffers
  uint8_t* out_dev = nullptr;
  uint32_t n = 0;
  uint32_t* LF = nullptr;
  uint32_t nLF = 0;
  uint32_t* freqs = nullptr;
  const BatchSpec* bs = nullptr;   // batch of blocks (block contract): the fields above come from *bs
  bwtc_cuda_runs* runs = nullptr;  // run statistics wanted (single block, block contract)
  int32_t* sa = nullptr;           // raw contract: the suffix array is emitted here (device; bwtc_cuda_divsufsort) ...
  int32_t* h_sa = nullptr;         // ... and copied to this host array once the block is finished (and verified)
  // ---- phase A
  uint32_t N = 0, bstride = 0, blk_bits = 0;
  bool sentinel_outside_alphabet = false;
  uint8_t last = 0;                // raw: T[N-1], the byte of the end-of-text row
  bool present[256];
  Round0Plan pl;
  const uint8_t* d_text = nullptr;
  uint8_t* d_dst = nullptr;
  EmitParams ep;
  uint64_t a_launches = 0, a_bytes = 0;  // kernel launches / algorithmic bytes of phase A
};

// Host wait for everything enqueued on `st` so far.  Default: sleep on a blocking-sync event — a waiting worker
// costs no host core, so `depth` workers per GPU times 8 ranks do not oversubscribe the box.  BWTC_SPIN_WAIT=1 spins.
int host_wait(bwtc_cuda_ctx* ctx, cudaStream_t st) {
  if (ctx->wait_mode == 1) {
    CK(ctx, cudaStreamSynchronize(st));
    return 0;
  }
  CK(ctx, cudaEventRecord(ctx->ev_sync, st));
  if (ctx->wait_mode == 2) {
    CK(ctx, cudaEventSynchronize(ctx->ev_sync));
    return 0;
  }
  // adaptive: a short busy poll catches the sub-100-us waits of a block running alone (a blocking-sync wake-up costs
  // ~0.3 ms on a virtualised host: measured, profiles/r02_experiments.md); after that the thread sleeps in ~50 us steps,
  // which costs a percent of a core however many blocks are in flight
  const auto t0 = std::chrono::steady_clock::now();
  for (;;) {
    const cudaError_t e = cudaEventQuery(ctx->ev_sync);
    if (e == cudaSuccess) return 0;
    if (e != cudaErrorNotReady) CK(ctx, e);
    const auto dt = std::chrono::steady_clock::now() - t0;
    if (dt > std::chrono::microseconds(ctx->poll_spin_us)) std::this_thread::sleep_for(std::chrono::microseconds(ctx->poll_sleep_us));
  }
}

// wait for one ring slot's copy (host side)
int ring_wait(bwtc_cuda_ctx* ctx, int slot) {
  if (!ctx->ring_busy[slot]) return 0;
  for (;;) {
    const cudaError_t e = cudaEventQuery(ctx->ev_ring[slot]);
    if (e == cudaSuccess) break;
    if (e != cudaErrorNotReady) CK(ctx, e);
    std::this_thread::yield();
  }
  ctx->ring_busy[slot] = false;
  return 0;
}

bool is_pinned_host(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// Device-side alias of a pinned host buffer (unified addressing), or nullptr if it is not mapped into the device's
// address space — then the copy engine is used.
uint8_t* mapped_alias(void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  if (a.type != cudaMemoryTypeHost) return nullptr;
  return static_cast<uint8_t*>(a.devicePointer);
}

int ensure_ring(bwtc_cuda_ctx* ctx) {
  if (ctx->h_ring) return 0;
  CK(ctx, cudaMallocHost((void**)&ctx->h_ring, RING_CHUNK * RING_SLOTS));
  CK(ctx, cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
  CK(ctx, cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
  for (int i = 0; i < RING_SLOTS; ++i)
    CK(ctx, cudaEventCreateWithFlags(&ctx->ev_ring[i], cudaEventBlockingSync | cudaEventDisableTiming));
  return 0;
}

// Host -> device.  Pinned source: one async copy on the kernel stream.  Pageable source: chunks through the pinned
// ring on the copy-in stream (the memcpy of chunk i+1 overlaps the DMA of chunk i); the kernel stream then waits
// for the last chunk.
int upload(bwtc_cuda_ctx* ctx, uint8_t* d_dst, const uint8_t* h_src, size_t n) {
  if (!n || (ctx->debug_skip_copies & 1)) return 0;
  if (is_pinned_host(h_src)) {
    CK(ctx, cudaMemcpyAsync(d_dst, h_src, n, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
  }
  if (ensure_ring(ctx)) return BWTC_CUDA_ECUDA;
  for (size_t off = 0; off < n; off += RING_CHUNK) {
    const size_t len = std::min(RING_CHUNK, n - off);
    const int slot = (int)(ctx->ring_next++ % RING_SLOTS);
    if (ring_wait(ctx, slot)) return BWTC_CUDA_ECUDA;  // (also across calls: the blocks of a batch are uploaded back to back)
    uint8_t* stage = ctx->h_ring + (size_t)slot * RING_CHUNK;
    memcpy(stage, h_src + off, len);
    CK(ctx, cudaMemcpyAsync(d_dst + off, stage, len, cudaMemcpyHostToDevice, ctx->s_in));
    CK(ctx, cudaEventRecord(ctx->ev_ring[slot], ctx->s_in));
    ctx->ring_busy[slot] = true;
  }
  CK(ctx, cudaEventRecord(ctx->ev_in, ctx->s_in));
  CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_in, 0));
  return 0;
}

// Device -> pageable host through the ring (blocking: returns when h_dst holds the bytes).  Everything enqueued on
// the kernel stream so far is waited for on the device (event), not by the host.
int download_staged(bwtc_cuda_ctx* ctx, uint8_t* h_dst, const uint8_t* d_src, size_t n) {
  if (!n) return 0;
  if (ensure_ring(ctx)) return BWTC_CUDA_ECUDA;
  CK(ctx, cudaEventRecord(ctx->ev_comp, ctx->stream));
  CK(ctx, cudaStreamWaitEvent(ctx->s_out, ctx->ev_comp, 0));
  for (int sl = 0; sl < RING_SLOTS; ++sl)
    if (ring_wait(ctx, sl)) return BWTC_CUDA_ECUDA;  // uploads that still read the ring
  const size_t nchunks = (n + RING_CHUNK - 1) / RING_CHUNK;
  const uint64_t base = ctx->ring_next;
  size_t issued = 0, done = 0;
  while (done < nchunks) {
    while (issued < nchunks && issued - done < (size_t)RING_SLOTS) {
      const int slot = (int)((base + issued) % RING_SLOTS);
      const size_t off = issued * RING_CHUNK, len = std::min(RING_CHUNK, n - off);
      CK(ctx, cudaMemcpyAsync(ctx->h_ring + (size_t)slot * RING_CHUNK, d_src + off, len, cudaMemcpyDeviceToHost, ctx->s_out));
      CK(ctx, cudaEventRecord(ctx->ev_ring[slot], ctx->s_out));
      ctx->ring_busy[slot] = true;
      ++issued;
    }
    const int slot = (int)((base + done) % RING_SLOTS);
    const size_t off = done * RING_CHUNK, len = std::min(RING_CHUNK, n - off);
    if (ring_wait(ctx, slot)) return BWTC_CUDA_ECUDA;
    memcpy(h_dst + off, ctx->h_ring + (size_t)slot * RING_CHUNK, len);
    ++done;
  }
  ctx->ring_next = base + nchunks;
  return 0;
}

// ---- phase A: input upload, reversed text + byte histogram, key-shape policy.  ONE host synchronisation (the plan
// needs the block's alphabet).  Nothing is written to the caller's arrays.
int64_t phase_input(bwtc_cuda_ctx* ctx, Job& J) {
  ctx->err[0] = 0;
  if (cudaSetDevice(ctx->device) != cudaSuccess) {
    set_err(ctx->err, "cudaSetDevice(%d) failed", ctx->device);
    return BWTC_CUDA_ECUDA;
  }
  const BatchSpec* bs = J.bs;
  J.bstride = bs ? bs->n0 + 1u : 0u;
  if (bs) {
    J.n = (bs->nblocks - 1u) * J.bstride + bs->n_last;  // N - 1
    J.nLF = bs->nLF;
    J.LF = bs->LF;
    J.freqs = bs->freqs;
  }
  const uint32_t n = J.n;
  const uint32_t N = J.block_mode ? n + 1 : n;
  J.N = N;
  // a context holds N = cap + 1 suffixes: a block of cap bytes plus its sentinel, or a raw text of cap + 1 bytes
  if (n > (J.block_mode ? (uint64_t)ctx->cap : (uint64_t)ctx->cap + 1)) {
    set_err(ctx->err, "%s of %u bytes exceeds context capacity %u", J.block_mode ? "block" : "raw text", n, ctx->cap);
    return BWTC_CUDA_ETOOBIG;
  }
  if (J.nLF < 1 || J.nLF > 256 || J.nLF > N || !J.LF) {
    set_err(ctx->err, "bad nLFpowers %u for %u suffixes", J.nLF, N);
    return BWTC_CUDA_EARG;
  }
  cudaStream_t st = ctx->stream;
  bwtc_cuda_stats& S = ctx->stats;
  memset(&S, 0, sizeof(S));
  S.n_suffixes = N;

  // ---- input
  const uint8_t* d_src = J.in_dev;
  const void** h_bptr = reinterpret_cast<const void**>(ctx->h_batch);
  uint32_t* h_bhist = reinterpret_cast<uint32_t*>(ctx->h_batch + MAX_BATCH * sizeof(void*));
  if (bs) {
    for (uint32_t k = 0; k < bs->nblocks; ++k) {
      const uint32_t nk = (k + 1 == bs->nblocks) ? bs->n_last : bs->n0;
      if (bs->on_device) {
        h_bptr[k] = bs->in[k];
      } else {
        if (upload(ctx, ctx->d_in + (size_t)k * bs->n0, static_cast<const uint8_t*>(bs->in[k]), nk)) return BWTC_CUDA_ECUDA;
        h_bptr[k] = ctx->d_in + (size_t)k * bs->n0;
      }
    }
    CK(ctx, cudaMemcpyAsync(ctx->d_bptr, h_bptr, bs->nblocks * sizeof(void*), cudaMemcpyHostToDevice, st));
    d_src = ctx->d_text;  // the policy sample reads the (reversed) concatenation
  } else if (!J.in_dev) {
    if (upload(ctx, ctx->d_in, J.h_in, n)) return BWTC_CUDA_ECUDA;
    d_src = ctx->d_in;
  }
  J.d_dst = (J.out_dev && !bs) ? J.out_dev : ctx->d_out;
  CK(ctx, cudaEventRecord(ctx->ev_begin, st));

  // ---- byte histogram (+ reversed, sentinel-terminated text in block mode)
  CK(ctx, cudaMemsetAsync(ctx->d_zero, 0, (size_t)(CTR_WORDS + HIST_WORDS) * 4, st));
  const int pgrid = ctx->sm_count * 8;
  if (bs) {
    const uint32_t padded_words = div_up((uint64_t)N + TEXT_PAD, 4);
    CK(ctx, cudaMemsetAsync(ctx->d_bhist, 0, (size_t)bs->nblocks * 256 * 4, st));
    const dim3 grid(std::max<uint32_t>(1u, div_up((uint32_t)pgrid, bs->nblocks)), bs->nblocks);
    k_prep_batch<<<grid, 256, 0, st>>>(reinterpret_cast<const uint8_t* const*>(ctx->d_bptr), bs->n0, bs->n_last, bs->nblocks,
                                       ctx->d_text, N, padded_words, ctx->d_bhist);
    J.d_text = ctx->d_text;
    S.algorithmic_bytes += 2ull * n + N;
  } else if (J.block_mode) {
    const uint32_t padded_words = div_up((uint64_t)N + TEXT_PAD, 4);
    k_prep_block<<<pgrid, 256, 0, st>>>(d_src, n, ctx->d_text, padded_words, ctx->d_hist());
    J.d_text = ctx->d_text;
    S.algorithmic_bytes += (uint64_t)n + N;
  } else {
    k_hist_bytes<<<pgrid, 256, 0, st>>>(d_src, N - 1, ctx->d_hist());
    J.d_text = d_src;
    S.algorithmic_bytes += (uint64_t)N;
  }
  CK(ctx, cudaGetLastError());
  S.kernel_launches++;
  double* d_pairs = reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(ctx->d_wtab) + (size_t)WS_SLOTS * 12);
  {  // sampled 8-byte-window collision statistics for the key-shape policy
    const uint32_t nbytes = J.block_mode ? n : N;
    uint32_t* d_cnt = reinterpret_cast<uint32_t*>(ctx->d_wtab + WS_SLOTS);
    CK(ctx, cudaMemsetAsync(ctx->d_wtab, 0xFF, (size_t)WS_SLOTS * 8, st));
    CK(ctx, cudaMemsetAsync(d_cnt, 0, (size_t)WS_SLOTS * 4 + 16, st));
    if (nbytes >= 8) {
      uint32_t stride = (nbytes - 7) >> 16;  // ~2^16 samples
      if (stride < 1) stride = 1;
      const uint32_t nsamp = (nbytes - 8) / stride + 1;
      k_window_sample<<<ctx->sm_count * 4, 256, 0, st>>>(d_src, nbytes, stride, nsamp, ctx->d_wtab, d_cnt);
      k_window_pairs<<<1, 1024, 0, st>>>(d_cnt, d_pairs);
      CK(ctx, cudaGetLastError());
      S.kernel_launches += 2;
    }
    CK(ctx, cudaMemcpyAsync(ctx->h_LF() + 256, d_pairs, 16, cudaMemcpyDeviceToHost, st));
  }
  if (bs) CK(ctx, cudaMemcpyAsync(h_bhist, ctx->d_bhist, (size_t)bs->nblocks * 256 * 4, cudaMemcpyDeviceToHost, st));
  else CK(ctx, cudaMemcpyAsync(ctx->h_hist(), ctx->d_hist(), 256 * 4, cudaMemcpyDeviceToHost, st));
  uint8_t* h_last = reinterpret_cast<uint8_t*>(ctx->h_LF() + 260);  // (behind the 16 bytes of pair statistics)
  if (!J.block_mode && !J.h_in) CK(ctx, cudaMemcpyAsync(h_last, d_src + (N - 1), 1, cudaMemcpyDeviceToHost, st));
  if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;

  uint64_t count[256];
  uint32_t npresent = 0;
  for (int c = 0; c < 256; ++c) {
    count[c] = 0;
    if (bs) for (uint32_t k = 0; k < bs->nblocks; ++k) count[c] += h_bhist[k * 256 + c];
    else count[c] = ctx->h_hist()[c];
    J.present[c] = count[c] != 0;
    npresent += J.present[c] ? 1u : 0u;
  }
  if (bs && npresent >= 256) return BATCH_NEEDS_SINGLE;
  // Block contract: the appended 0x00 only enters the alphabet if the block itself contains 0x00.  Otherwise
  // it is a true sentinel: it gets code 0 like the padding past the end, and the "window ran past the end"
  // rule of the round-0 re-rank starts one position earlier (DESIGN.md §3.2) — a 4-letter alphabet then packs
  // into 2 bits per character instead of 3.  A batch reserves code 0 for its sentinels instead (§3.6).
  J.sentinel_outside_alphabet = false;
  J.blk_bits = 0;
  if (bs) {
    J.blk_bits = std::max<uint32_t>(1u, (uint32_t)ceil_log2_u64(bs->nblocks));
  } else if (J.block_mode) {
    if (!J.present[0]) J.sentinel_outside_alphabet = true;
  } else {
    const uint8_t last = J.h_in ? J.h_in[N - 1] : *h_last;
    J.last = last;
    J.present[last] = true;
    count[last] += 1;
  }
  double pair_stats[2];  // [0] colliding pairs among the sampled 8-byte windows, [1] samples
  memcpy(pair_stats, ctx->h_LF() + 256, 16);
  plan_round0(ctx, count, J.present, N, pair_stats, &J.pl, J.blk_bits);
  if (bs) { J.pl.pp.nblocks = bs->nblocks; J.pl.pp.stride = J.bstride; }
  J.ep.nblocks = bs ? bs->nblocks : 1u;
  J.ep.stride = J.bstride;
  J.ep.text = J.d_text;
  J.ep.out = J.d_dst;
  J.ep.lastch = ctx->d_LF + LF_PARK;
  J.ep.N = N;
  J.ep.block_mode = J.block_mode ? 1 : 0;
  J.ep.sa = J.sa;
  S.sigma = J.pl.sigma;
  S.bits_per_char = J.pl.bits;
  S.chars_round0 = J.pl.chars;
  S.key_bytes_round0 = J.pl.keybytes;
  J.a_launches = S.kernel_launches;
  J.a_bytes = S.algorithmic_bytes;
  return 0;
}

int verify_forward(bwtc_cuda_ctx* ctx, const Job& J);
int verify_sa(bwtc_cuda_ctx* ctx, const Job& J);

// ---- phase B: round 0, the device-controlled ladder of sort-free rounds, host-driven global radix rounds where
// groups are large, final extraction, result copies.  Works from ctx->d_text only, so it can be repeated (with ticket
// tile ids) after a look-back watchdog without the caller's input.
int64_t phase_sort(bwtc_cuda_ctx* ctx, Job& J) {
  ctx->lb_watchdog = 0;
  if (cudaSetDevice(ctx->device) != cudaSuccess) {
    set_err(ctx->err, "cudaSetDevice(%d) failed", ctx->device);
    return BWTC_CUDA_ECUDA;
  }
  cudaStream_t st = ctx->stream;
  bwtc_cuda_stats& S = ctx->stats;
  const BatchSpec* bs = J.bs;
  const uint32_t N = J.N, n = J.n;
  const Round0Plan& pl = J.pl;
  const EmitParams& ep = J.ep;
  const uint8_t* d_text = J.d_text;
  PassTimer pt{ctx};
  // a repeated phase B starts its statistics over (phase A's launches and bytes are kept)
  S.kernel_launches = J.a_launches;
  S.algorithmic_bytes = J.a_bytes;
  S.sort_bytes = S.sort0_bytes = 0;
  S.sort_launches = S.sort0_launches = 0;
  CK(ctx, cudaMemsetAsync(ctx->d_zero, 0, (size_t)CTR_STICKY * 4, st));  // sticky control words (CTR_ERR)
  CK(ctx, cudaMemsetAsync(ctx->d_state, 0, sizeof(LadderState), st));
  CK(ctx, cudaMemsetAsync(ctx->d_LF + LF_PARK, 0, (size_t)(LF_WORDS - LF_PARK) * 4, st));  // parked hole bytes

  // ---- round 0: pack keys (+ all digit histograms), sort, re-rank
  const uint32_t rs_tile0 = pl.keybytes == 4 ? RS_TILE32 : RS_TILE64;
  const uint32_t all0 = (1u << pl.npass) - 1u;
  if (zero_round_state(ctx, N, N, rs_tile0, all0, pl.rb)) return BWTC_CUDA_ECUDA;
  {
    const uint32_t ptiles = div_up(N, AUX_TILE);
    const int grid = (int)(ptiles < (uint32_t)(ctx->sm_count * 4) ? ptiles : (uint32_t)(ctx->sm_count * 4));
    // One representative digit per phase class is counted by k_pack_round0; the others are derived (k_hist_derive).
    uint32_t hist_mask = 0;
    DeriveParams dp;
    dp.count = 0;
    // (digit positions in the coordinates of the c exact characters: the key carries pl.rbits partial bits below them)
    const uint32_t keybits = pl.chars * pl.bits;
    const uint32_t rbits = pl.rbits;
    uint32_t regular_mask = 0;  // digits that lie entirely inside the exact characters
    for (uint32_t p = 0; p < pl.npass; ++p) {
      int rep = -1;
      const uint32_t rb = pl.rb;
      const bool full_p = (rb * p >= rbits) && (rb * p - rbits + rb <= keybits);
      if (full_p) regular_mask |= 1u << p;
      if (full_p && N > 64 && !bs)  // (a batch counts every digit directly: block numbers sit above the characters)
        for (uint32_t r = 0; r < p; ++r)
          if (((hist_mask >> r) & (regular_mask >> r) & 1u) && (rb * (p - r)) % pl.bits == 0) { rep = (int)r; break; }
      if (rep < 0) {
        hist_mask |= 1u << p;
      } else {
        dp.p[dp.count] = (uint8_t)p;
        dp.r[dp.count] = (uint8_t)rep;
        dp.t[dp.count] = (uint8_t)(pl.rb * (p - (uint32_t)rep) / pl.bits);
        dp.count++;
      }
    }
    // Gram mode (6- and 3-bit codes): one 4096-bin histogram of the keys' low 12 bits, every digit histogram projected
    // from it (k_hist_from_gram) — one shared-memory atomic per key instead of one per counted digit.
    GramParams gp;
    gp.npass = 0;
    bool use_gram = ctx->use_gram && !bs && N > 64 && (pl.bits == 6 || pl.bits == 3) && keybits >= (uint32_t)GRAM_BITS;
    if (use_gram) {
      const uint32_t W = (uint32_t)GRAM_BITS / pl.bits;
      for (uint32_t p = 0; p < pl.npass && use_gram; ++p) {
        uint32_t u, sft;
        gp.next[p] = 0;
        if (pl.rb * p < rbits) {  // the lowest digit reaches into the partial character: window of the following suffix
          if (p != 0) use_gram = false;
          u = 0;
          sft = pl.bits - rbits;
          gp.next[p] = 1;
          if (sft + pl.rb > (uint32_t)GRAM_BITS) use_gram = false;
        } else {
          const uint32_t lo = pl.rb * p - rbits;
          u = std::min<uint32_t>(lo / pl.bits, pl.chars - W);
          sft = lo - pl.bits * u;
          // the digit must lie inside the 12 bits above bit (bits * u), or run past the top of the key (zeros there)
          if (sft + pl.rb > (uint32_t)GRAM_BITS && lo + pl.rb <= keybits) use_gram = false;
        }
        if (sft >= 32u) use_gram = false;
        gp.u[p] = (uint8_t)u;
        gp.s[p] = (uint8_t)sft;
      }
      gp.npass = pl.npass;
    }
    uint32_t* gram = use_gram ? ctx->d_hist() + GRAM_OFF : nullptr;
    if (use_gram) { hist_mask = 0; dp.count = 0; }
    if (pl.keybytes == 4) {
      k_pack_round0<uint32_t><<<grid, 256, 0, st>>>(d_text, N, static_cast<uint32_t*>(ctx->d_keys[0]), pl.pp,
                                                     ctx->d_hist(), hist_mask, ptiles, pl.rb, gram);
      if (dp.count) k_hist_derive<uint32_t><<<dp.count, 256, 0, st>>>(d_text, N, pl.pp, dp, ctx->d_hist(), pl.rb);
      if (use_gram) k_hist_from_gram<uint32_t><<<gp.npass, 256, 0, st>>>(d_text, N, pl.pp, gp, gram, ctx->d_hist(), pl.rb);
    } else {
      k_pack_round0<unsigned long long><<<grid, 256, 0, st>>>(d_text, N, static_cast<unsigned long long*>(ctx->d_keys[0]),
                                                               pl.pp, ctx->d_hist(), hist_mask, ptiles, pl.rb, gram);
      if (dp.count) k_hist_derive<unsigned long long><<<dp.count, 256, 0, st>>>(d_text, N, pl.pp, dp, ctx->d_hist(), pl.rb);
      if (use_gram)
        k_hist_from_gram<unsigned long long><<<gp.npass, 256, 0, st>>>(d_text, N, pl.pp, gp, gram, ctx->d_hist(), pl.rb);
    }
    if (dp.count || use_gram) S.kernel_launches++;
    CK(ctx, cudaGetLastError());
    S.kernel_launches++;
    S.algorithmic_bytes += (uint64_t)N + (uint64_t)N * pl.keybytes;
  }
  // every digit pass of the round runs: a constant digit makes its pass a (stable) identity permutation, and
  // finding that out would cost a host synchronisation per block
  const uint32_t mask0 = all0;
  int cur = 0;
  uint32_t pdone = 0;
  int rc;
  // When the id and one character code fit a 32-bit payload together, the first pass stores the code of the
  // character preceding each suffix above the id: the round-0 BWT emission then needs no text gather.
  uint32_t id_bits = (uint32_t)ceil_log2_u64((uint64_t)N);
  if (id_bits < 1) id_bits = 1;
  const bool pack_pred = ctx->use_pack_pred && (id_bits + pl.bits <= 32) && (mask0 & 1u);
  const uint32_t topshift = (pl.chars - 1) * pl.bits + pl.rbits;
  const uint32_t pred_mask = (1u << pl.bits) - 1u;  // (a batch key carries the block number above the characters)
  // No spare id bits (byte alphabets above 16 MiB) and a text too large for an L2-resident gather at emission time:
  // the predecessor codes travel as a one-byte payload array instead.
  const bool aux_pred = !pack_pred && ctx->aux_min_suffixes && N >= ctx->aux_min_suffixes && (mask0 & 1u) && !bs;
  if (pl.keybytes == 4)
    rc = run_sort<uint32_t, RS_IPT32>(ctx, N, mask0, true, N - 1, &cur, &pt, &pdone, pack_pred ? id_bits : 0u, topshift,
                                      pred_mask, aux_pred);
  else
    rc = run_sort<unsigned long long, RS_IPT64>(ctx, N, mask0, true, N - 1, &cur, &pt, &pdone, pack_pred ? id_bits : 0u,
                                                topshift, pred_mask, aux_pred, pl.rb);
  if (rc) return rc;
  const size_t round0_events = pt.used;
  S.sort0_launches = S.sort_launches;
  S.sort0_bytes = S.sort_bytes;
  S.live[0] = N;
  S.passes[0] = pdone;
  S.prefix_len[0] = 0;
  S.rounds = 1;
  // ---- lazy ranks? (DESIGN.md §3.9)  The rank scatter of round 0 — a random 4-byte write per suffix — is 20-35% of a block,
  // but after round 0 only the ranks of suffixes that are still in a group are ever refined, and a singleton's rank is simply
  // its position in the sorted key array.  If few suffixes will stay in groups, rank[] is written for those only; the
  // segmented rounds order group members by cmp (round-0 key, then rank where it is stored) and need no integer rank, the
  // tail (k_small_rounds, k_finish) looks the few ranks it needs up in the retained sorted keys (rank_lookup).
  bool lazy = false;
  const uint32_t keybits0 = pl.chars * pl.bits + pl.rbits;
  if (ctx->use_lazy && !bs && !dbg_any(ctx) && N >= 64 && keybits0 >= 1) {
    // The decision needs no extra measurement.  For an i.i.d.-like source (DNA, random bytes) the key-shape policy has
    // already predicted the fraction of suffixes still tied after round 0, L(c) = 1 - exp(-N 2^(-H0 c)) — it matches the
    // measured live fractions to three digits (DNA 64 MiB: 0.0156 / 0.0155; random 256 MiB: 0.0606 / 0.0606).  For a source
    // with memory the 8-gram sample tells text (a few other positions share a position's 8-gram: Markov 32 MiB 3.0, 3% live
    // after its 10.7-character keys) from repeats (thousands: the 4 KiB-seed block keeps ~all suffixes tied through global
    // radix rounds and would only pay the materialising fallback).  The 8-gram sample says nothing about how much a key
    // longer than 8 characters separates, so a block with memory also needs keys of at least LAZY_MIN_CHARS characters
    // (codes of <= 6 bits): the same Markov text as a 65-symbol raw text (7-bit codes, 9-character keys) left more or
    // larger groups after round 0 than the segmented rounds take and fell back.  Segmented rounds are what makes lazy ranks cheap, so a block with memory
    // goes lazy only where they run.  A wrong prediction only costs time: the fallback below is exact.
    constexpr uint32_t LAZY_MIN_CHARS = 10;
    const bool memory_ok = ctx->use_seg && pl.chars >= LAZY_MIN_CHARS && pl.repeats <= ctx->lazy_max_repeats;
    lazy = ctx->use_lazy >= 2 ||
           (N >= ctx->lazy_min_suffixes && (pl.has_memory ? memory_ok : pl.live_pred <= ctx->lazy_max_live));
  }
  const uint32_t tbits = std::min<uint32_t>(KTAB_BITS, keybits0);
  const uint32_t lazy_cap = N / 6;  // the lists of lazy mode live in six slices of d_scat
  {
    RerankParams rp;
    rp.m = N;
    {
      const uint32_t text_end = J.sentinel_outside_alphabet ? N - 1 : N;  // windows reaching text_end are unique
      const uint32_t wchars = pl.chars + (pl.rbits ? 1u : 0u);  // characters a key looks at (the partial one included)
      rp.short_thresh = wchars > text_end ? 0u : text_end - wchars + 1u;
    }
    rp.lo_bits = 0;
    rp.lazy = lazy ? 1u : 0u;
    rp.livebits = ctx->d_livebits;
    rp.ktab = ctx->d_ktab;
    rp.tshift = keybits0 - tbits;
    if (lazy) {
      CK(ctx, cudaMemsetAsync(ctx->d_livebits, 0, ((size_t)N / 32 + 4) * 4, st));
      CK(ctx, cudaMemsetAsync(ctx->d_ktab, 0xFF, ((size_t)(1u << tbits) + 2) * 4, st));
      LookupParams& L = *ctx->h_lookup;
      L.enabled = 1;
      L.keybytes = pl.keybytes;
      L.sorted_keys = ctx->d_keys[cur];
      L.ktab = ctx->d_ktab;
      L.livebits = ctx->d_livebits;
      L.text = d_text;
      L.N = N;
      L.bits = pl.bits;
      L.chars = pl.chars;
      L.rbits = pl.rbits;
      L.tshift = keybits0 - tbits;
      memcpy(L.lut, pl.pp.lut, 256);
      CK(ctx, cudaMemcpyAsync(ctx->d_lookup, ctx->h_lookup, sizeof(LookupParams), cudaMemcpyHostToDevice, st));
    }
    S.flags = (ctx->static_tiles ? 0u : 1u) | (bs ? 2u : 0u) | (pack_pred ? 4u : 0u) | (aux_pred ? 8u : 0u) | (lazy ? 16u : 0u) |
              (J.sa ? 256u : 0u);
    rp.packed = pack_pred ? 1u : (aux_pred ? 2u : 0u);
    rp.pred_aux = ctx->d_aux[cur];
    rp.id_bits = pack_pred ? id_bits : 31u;
    rp.id_mask = pack_pred ? (uint32_t)((1ull << id_bits) - 1ull) : 0xFFFFFFFFu;
    memset(rp.decode, 0, sizeof(rp.decode));
    for (int c = 0; c < 256; ++c)
      if (J.present[c]) rp.decode[pl.pp.lut[c]] = (uint8_t)c;
    uint32_t* snr = reinterpret_cast<uint32_t*>(ctx->d_keys[cur ^ 1]);
    if (pl.keybytes == 4) rc = launch_rerank<uint32_t, true>(ctx, cur, N, N, rp, ep, snr, snr + N, lazy);
    else rc = launch_rerank<unsigned long long, true>(ctx, cur, N, N, rp, ep, snr, snr + N, lazy);
    if (rc) return rc;
    S.algorithmic_bytes += (uint64_t)N * (pl.keybytes + 4) + (lazy ? 0ull : (uint64_t)N * 4);
    if (lazy) {
      const uint32_t entries = 1u << tbits, nchunks = div_up(entries, KTAB_CHUNK);
      uint32_t* cmin = ctx->d_bhist;  // <= 256 words of the (idle) per-block histogram area
      k_ktab_chunkmin<<<nchunks, 256, 0, st>>>(ctx->d_ktab, entries, cmin);
      k_ktab_fill<<<nchunks, 256, 0, st>>>(ctx->d_ktab, entries, N, cmin, nchunks);
      CK(ctx, cudaGetLastError());
      S.kernel_launches += 2;
    }
    ctx->rr0 = rp;  // (kept for the fallback out of lazy mode)
  }
  // six u32[N] work arrays: halves of the two key buffers and the two id buffers
  PoolPtrs pool;
  pool.p[0] = reinterpret_cast<uint32_t*>(ctx->d_keys[0]);
  pool.p[1] = reinterpret_cast<uint32_t*>(ctx->d_keys[0]) + N;
  pool.p[2] = reinterpret_cast<uint32_t*>(ctx->d_keys[1]);
  pool.p[3] = reinterpret_cast<uint32_t*>(ctx->d_keys[1]) + N;
  pool.p[4] = ctx->d_idx[0];
  pool.p[5] = ctx->d_idx[1];
  const PoolPtrs norm = pool;  // (the staging slots of k_rerank are always halves of the idle key buffer)
  if (lazy) {  // the sorted keys (d_keys[cur]) must survive: lists, next lists and rank updates live in six slices of d_scat
    for (int q = 0; q < 6; ++q) pool.p[q] = ctx->d_scat + (size_t)q * lazy_cap;
  }
  const LookupParams* lkp = lazy ? ctx->d_lookup : nullptr;
  ctx->last_cur = cur;
  uint32_t m_prev = N;       // records of the last global sort = extent of the k_rerank staging slots
  uint32_t m_bound = N;      // upper bound of the live count (it never grows)
  uint64_t h_next = pl.chars;
  auto sel_of = [&lazy](int c) { return lazy ? 0x10u : ((uint32_t)(2 * c) | ((uint32_t)(2 * c + 1) << 4)); };
  k_commit_sort<<<1, 1, 0, st>>>(ctx->d_state, ctx->d_ctrl(), (uint32_t)std::min<uint64_t>(h_next, 0x7FFFFFFFull), sel_of(cur),
                                 0xFFFFFFFFu, 1u, lazy ? lazy_cap : 0xFFFFFFFFu);
  S.kernel_launches++;

  // Concatenate the per-tile chunks k_rerank staged (in d_keys[cur^1]) into compact lists in d_keys[cur], whose
  // sorted keys are dead by now.  Tile order is kept, so every group stays contiguous.  speculative: the gather
  // runs only if the device-side state says the next step consumes the lists.
  auto make_lists = [&](bool speculative) -> int {
    const uint32_t tiles = div_up(m_prev, AUX_TILE);
    k_scan_tile_counts<<<1, 1024, 0, st>>>(ctx->d_tilecnt, ctx->d_tilecnt + ctx->max_aux_tiles, tiles);
    k_gather_chunks<<<tiles, 256, 0, st>>>(norm.p[2 * (cur ^ 1)], norm.p[2 * (cur ^ 1) + 1], ctx->d_tilecnt,
                                           ctx->d_tilecnt + ctx->max_aux_tiles, AUX_TILE, lazy ? pool.p[0] : norm.p[2 * cur],
                                           lazy ? pool.p[1] : norm.p[2 * cur + 1], speculative ? ctx->d_state : nullptr,
                                           ctx->d_ctrl());
    CK(ctx, cudaGetLastError());
    S.kernel_launches += 2;
    return 0;
  };

  // Result copies that need no host staging: pinned host buffers and device buffers.  Enqueued speculatively behind the
  // first ladder chunk (a block whose later rounds are all sort-free then completes with one host wait); repeated at
  // the end if the block was not finished by then.
  const bool direct_out = bs ? (bs->on_device || is_pinned_host(bs->out[0]))
                             : (J.out_dev != nullptr || (J.block_mode && J.h_out && is_pinned_host(J.h_out)));
  // verification (DESIGN.md §3.10): the caller's host and batch outputs are written only after the check word is read
  const bool verify = ctx->verify && !ctx->debug_max_rounds;
  uint32_t* h_bLF = reinterpret_cast<uint32_t*>(ctx->h_batch + MAX_BATCH * sizeof(void*)) + MAX_BATCH * 256;
  auto enqueue_direct_out = [&]() -> int {
    if (bs) {
      for (uint32_t k = 0; k < bs->nblocks; ++k) {  // block k's BWT bytes are out[k*stride .. k*stride + n_k)
        const uint32_t nk = (k + 1 == bs->nblocks) ? bs->n_last : bs->n0;
        CK(ctx, cudaMemcpyAsync(bs->out[k], ctx->d_out + (size_t)k * J.bstride, nk,
                                bs->on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
      }
    } else if (!J.out_dev && !(ctx->debug_skip_copies & 2)) {
      uint8_t* alias = ctx->d2h_kernel ? mapped_alias(J.h_out) : nullptr;
      if (alias) {
        k_copy_out<<<ctx->d2h_ctas, 256, 0, st>>>(ctx->d_out, alias, n, ctx->d_state, ctx->d_ctrl());
        CK(ctx, cudaGetLastError());
        S.kernel_launches++;
      } else {
        CK(ctx, cudaMemcpyAsync(J.h_out, ctx->d_out, n, cudaMemcpyDeviceToHost, st));
      }
    }
    return 0;
  };

  const int lo_bits = (int)ceil_log2_u64((uint64_t)N + 1);  // rank[i+h] + 1 in [0, N]
  // high part = (rank of the group head) >> 1 (k_build_keys): heads of live groups are <= N - 2
  const int hi_bits = N > 3 ? (int)ceil_log2_u64((((uint64_t)N - 2) >> 1) + 1) : 1;
  uint32_t npassd = div_up((uint64_t)(lo_bits + hi_bits), 8), rbd = 8;
  if (ctx->use_radix9 && div_up((uint64_t)(lo_bits + hi_bits), 9) < npassd) {  // 9-bit digits when they save a pass
    npassd = div_up((uint64_t)(lo_bits + hi_bits), 9);
    rbd = 9;
  }
  const uint32_t maskd = (1u << npassd) - 1u;
  bool lists_pending = true, first_chunk = true, out_enqueued = false, finished = false;
  // lean chunk: behind a global radix round whose groups were still far above the segmented-round limit nothing sort-free
  // is enqueued speculatively (it would only be skipped on the device): commit, k_finish (error word), state copy, wait
  bool lean = false;
  constexpr uint32_t LEAN_MAXGROUP = 8u * SEG_MAXGROUP;
  uint32_t nlog_seen = 0;
  const uint32_t dbg = ctx->debug_max_rounds;
  for (;;) {
    // ---- one ladder chunk: [lists] [K x (segmented round, rank update, commit)] [tail] [finish] [copies]
    const bool chunk_built_lists = lists_pending && !lean;
    if (!(dbg && S.rounds >= dbg) && !lean) {
      if (lists_pending) {
        if (make_lists(true)) return BWTC_CUDA_ECUDA;
        lists_pending = false;
      }
      const int K = dbg ? 1 : (first_chunk ? ctx->ladder_first : ctx->ladder_more);
      for (int k = 0; k < K && ctx->use_seg; ++k) {
        // persistent grid; the first round behind a sort is the big one, later (often skipped) ones get a leaner grid
        const uint32_t per_sm = (k == 0) ? 12u : 4u;
        const uint32_t seg_grid = std::max<uint32_t>(1u, std::min<uint32_t>(div_up(m_bound, SEG_T), (uint32_t)ctx->sm_count * per_sm));
        if (ep.sa) {
          if (lkp) k_seg_round<true, true><<<seg_grid, 256, 0, st>>>(ctx->d_state, pool, ctx->d_rank, N, ep, ctx->d_ctrl(), lkp);
          else k_seg_round<false, true><<<seg_grid, 256, 0, st>>>(ctx->d_state, pool, ctx->d_rank, N, ep, ctx->d_ctrl(), nullptr);
        } else {
          if (lkp) k_seg_round<true><<<seg_grid, 256, 0, st>>>(ctx->d_state, pool, ctx->d_rank, N, ep, ctx->d_ctrl(), lkp);
          else k_seg_round<false><<<seg_grid, 256, 0, st>>>(ctx->d_state, pool, ctx->d_rank, N, ep, ctx->d_ctrl(), nullptr);
        }
        k_apply_ranks<<<ctx->sm_count * 8, 256, 0, st>>>(ctx->d_state, pool, ctx->d_ctrl(), ctx->d_rank);
        k_commit_seg<<<1, 1, 0, st>>>(ctx->d_state, ctx->d_ctrl());
        S.kernel_launches += 3;
      }
      if (!dbg) {
        if (ep.sa) k_small_rounds<true><<<1, 1024, 0, st>>>(ctx->d_state, pool, ctx->d_rank, N, ep, ctx->d_ctrl(), lkp);
        else k_small_rounds<<<1, 1024, 0, st>>>(ctx->d_state, pool, ctx->d_rank, N, ep, ctx->d_ctrl(), lkp);
        S.kernel_launches++;
      }
      CK(ctx, cudaGetLastError());
    }
    // final extraction: pidx, LFpowers, hole fill (returns early on the device while suffixes are still live)
    if (bs)
      k_finish_batch<<<bs->nblocks, 256, 0, st>>>(ctx->d_rank, N, J.bstride, bs->nblocks, J.d_dst, ctx->d_LF, bs->nLF, bs->nLF_last,
                                                  ctx->d_LF + LF_PARK, ctx->d_state, ctx->d_ctrl());
    else
      k_finish<<<1, 256, 0, st>>>(ctx->d_rank, d_text, N, J.d_dst, J.block_mode ? 1 : 0, ctx->d_LF, J.nLF, ctx->d_LF + LF_PARK,
                                  ctx->d_state, ctx->d_ctrl(), lkp);
    CK(ctx, cudaGetLastError());
    S.kernel_launches++;
    if (J.runs && !bs && J.block_mode) {
      // run statistics of the (finished) output: symbols -> d_aux[0], start positions -> d_scat, both idle by now; tile
      // counts in the look-back status area (cleared again before any later digit pass uses it)
      const uint32_t rtiles = div_up(n, RUN_TILE);
      uint32_t* rcnt = status_rows(ctx, 0);
      uint32_t* rexcl = rcnt + rtiles;
      const uint32_t cap_dev = std::min<uint32_t>(J.runs->capacity, n);
      k_run_count<<<rtiles, 256, 0, st>>>(J.d_dst, n, rcnt, ctx->d_state);
      k_scan_tile_counts<<<1, 1024, 0, st>>>(rcnt, rexcl, rtiles);
      k_run_emit<<<rtiles, 256, 0, st>>>(J.d_dst, n, rcnt, rexcl, rtiles, cap_dev, ctx->d_aux[0], ctx->d_scat, &ctx->d_state->nruns,
                                         ctx->d_state);
      CK(ctx, cudaGetLastError());
      S.kernel_launches += 3;  // (queued in every chunk; they return at once in all but the one that finishes the block)
    }
    CK(ctx, cudaEventRecord(ctx->ev_end, st));
    CK(ctx, cudaMemcpyAsync(ctx->h_state, ctx->d_state, sizeof(LadderState), cudaMemcpyDeviceToHost, st));
    if (bs) CK(ctx, cudaMemcpyAsync(h_bLF, ctx->d_LF, (size_t)bs->nblocks * 256 * 4, cudaMemcpyDeviceToHost, st));
    else CK(ctx, cudaMemcpyAsync(ctx->h_LF(), ctx->d_LF, J.nLF * 4, cudaMemcpyDeviceToHost, st));
    if (first_chunk && direct_out && !dbg && !verify) {
      if (enqueue_direct_out()) return BWTC_CUDA_ECUDA;
      out_enqueued = true;
    }
    if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
    const LadderState& H = *ctx->h_state;
    if (H.err == 4u) {
      set_err(ctx->err, "segmented round met a group above its limit (internal error)");
      return BWTC_CUDA_EINTERNAL;
    }
    if (H.err == 5u) {
      set_err(ctx->err, "k_build_keys emitted a record count that differs from the live count (internal error)");
      return BWTC_CUDA_EINTERNAL;
    }
    if (H.err == 3u) {
      set_err(ctx->err, "tail refinement kernel did not converge");
      return BWTC_CUDA_EINTERNAL;
    }
    if (H.err || (ctx->debug_fake_watchdog && ctx->static_tiles)) {
      set_err(ctx->err, "look-back watchdog fired (code %u, round %u)", H.err, S.rounds);
      ctx->lb_watchdog = 1;
      return BWTC_CUDA_EINTERNAL;
    }
    // rounds the device executed in this chunk
    for (uint32_t i = nlog_seen; i < H.nlog && i < (uint32_t)LADDER_LOG; ++i) {
      const uint32_t r = S.rounds;
      if (chunk_built_lists && i == nlog_seen) S.algorithmic_bytes += (uint64_t)H.log_m[i] * 16;  // k_gather_chunks
      if (r < BWTC_CUDA_MAX_ROUNDS) {
        S.live[r] = H.log_m[i];
        S.passes[r] = 0;
        S.prefix_len[r] = H.log_h[i];
        S.rounds = r + 1;
      }
      S.algorithmic_bytes += (uint64_t)H.log_m[i] * (H.log_kind[i] == 1u ? 32u : 24u);
    }
    nlog_seen = H.nlog;
    first_chunk = false;
    if (H.m == 0) { finished = true; break; }
    out_enqueued = false;  // the speculative copies ran before the block was complete: repeat them at the end
    if (lazy && !H.lists) {
      // Out of lazy mode: more suffixes stayed in groups than the small list pool holds, or groups are large (a global
      // radix round scans rank[] in text order and needs every rank).  Materialise the singletons' ranks from the sorted
      // records of round 0 (still intact), then carry on with the full-rank path; nothing else has run in between.
      RerankParams rp = ctx->rr0;
      rp.lazy = 2u;
      CK(ctx, cudaMemsetAsync(ctx->d_tstate(), 0, (size_t)rerank_launches(ctx, N, N) * ctx->max_aux_tiles * 8, st));
      CK(ctx, cudaMemsetAsync(ctx->d_ctrl() + CTR_PASS0, 0, (size_t)(CTR_WORDS - CTR_PASS0) * 4, st));  // tile tickets
      uint32_t* snr = reinterpret_cast<uint32_t*>(ctx->d_keys[cur ^ 1]);
      lazy = false;  // (sel_of and the pools below now mean the full-rank layout)
      if (pl.keybytes == 4) rc = launch_rerank<uint32_t, true>(ctx, cur, N, N, rp, ep, snr, snr + N, false, true);
      else rc = launch_rerank<unsigned long long, true>(ctx, cur, N, N, rp, ep, snr, snr + N, false, true);
      if (rc) return rc;
      S.algorithmic_bytes += (uint64_t)N * (pl.keybytes + 4) + (uint64_t)N * 4;
      S.flags |= 32u;  // lazy ranks were abandoned for this block
      pool = norm;
      lkp = nullptr;
      lean = true;  // the lists (if the next step wants them) are built below from the intact staging
      lists_pending = true;
    }
    if (lean) {
      lean = false;
      if (H.m <= (uint32_t)SMALL_MAX || (ctx->use_seg && H.maxgroup <= (uint32_t)SEG_MAXGROUP)) {
        // the groups collapsed after all: build the lists now and run a normal ladder chunk
        if (make_lists(false)) return BWTC_CUDA_ECUDA;
        k_mark_lists<<<1, 1, 0, st>>>(ctx->d_state, sel_of(cur));
        CK(ctx, cudaGetLastError());
        S.kernel_launches++;
        S.algorithmic_bytes += (uint64_t)H.m * 16;
        lists_pending = false;
        m_bound = H.m;
        continue;
      }
    }
    if (dbg && S.rounds >= dbg) break;
    const uint32_t m = H.m;
    m_bound = m;
    if (S.rounds >= BWTC_CUDA_MAX_ROUNDS - 1 || (uint64_t)H.h >= 2ull * N + 2) {
      set_err(ctx->err, "prefix doubling did not converge (round %u, h %u, live %u)", S.rounds, H.h, m);
      return BWTC_CUDA_EINTERNAL;
    }
    if (ctx->use_seg && H.lists && H.maxgroup <= (uint32_t)SEG_MAXGROUP) continue;  // more segmented rounds than were enqueued
    if (m <= (uint32_t)SMALL_MAX && !dbg) {
      set_err(ctx->err, "internal: tail kernel skipped %u live suffixes", m);
      return BWTC_CUDA_EINTERNAL;
    }

    // ---- global radix round (large groups: repetitive input), host-driven
    const uint32_t r = S.rounds;
    const uint32_t h32 = H.h;
    const bool from_list = ((uint64_t)m * 8 <= (uint64_t)N);
    const bool have_lists = H.lists != 0;
    if (have_lists && H.sel != sel_of(cur)) {  // group sizes never grow, so a segmented round is never followed by a global sort
      set_err(ctx->err, "internal: global sort requested after a segmented round (maxgroup %u)", H.maxgroup);
      return BWTC_CUDA_EINTERNAL;
    }
    if (zero_round_state(ctx, N, m, RS_TILE64, maskd, rbd)) return BWTC_CUDA_ECUDA;
    uint32_t expect_cursor = 0xFFFFFFFFu;
    if (from_list) {
      if (!have_lists) {
        if (make_lists(false)) return BWTC_CUDA_ECUDA;
        S.algorithmic_bytes += (uint64_t)m * 16;
      }
      // few live suffixes: gather-build from the id list (in d_keys[cur]) into the other buffer pair
      const int tb = cur ^ 1;
      const uint32_t bt = div_up(m, 256);
      const int grid = (int)(bt < (uint32_t)(ctx->sm_count * 8) ? bt : (uint32_t)(ctx->sm_count * 8));
      k_build_from_list<<<grid, 256, 0, st>>>(pool.p[2 * cur + 1], m, ctx->d_rank, N, h32, lo_bits,
                                              static_cast<unsigned long long*>(ctx->d_keys[tb]), ctx->d_idx[tb],
                                              ctx->d_hist(), (int)npassd, ctx->d_ctrl(), rbd);
      CK(ctx, cudaGetLastError());
      S.kernel_launches++;
      S.algorithmic_bytes += (uint64_t)m * (4 + 8 + 12);
      cur = tb;
    } else {
      const uint32_t btiles = div_up(N, AUX_TILE);
      const int grid = (int)(btiles < (uint32_t)(ctx->sm_count * 8) ? btiles : (uint32_t)(ctx->sm_count * 8));
      k_build_keys<<<grid, 256, 0, st>>>(ctx->d_rank, N, h32, lo_bits, static_cast<unsigned long long*>(ctx->d_keys[0]),
                                         ctx->d_idx[0], ctx->d_ctrl(), ctx->d_hist(), (int)npassd, btiles, rbd);
      CK(ctx, cudaGetLastError());
      S.kernel_launches++;
      S.algorithmic_bytes += (uint64_t)N * 4 + (uint64_t)m * 12;
      cur = 0;
      expect_cursor = m;
    }
    rc = run_sort<unsigned long long, RS_IPT64>(ctx, m, maskd, false, 0, &cur, &pt, &pdone, 0, 0, 0xFFFFFFFFu, false, rbd);
    if (rc) return rc;
    {
      RerankParams rp;
      rp.m = m;
      rp.short_thresh = 0;
      rp.lo_bits = lo_bits;
      rp.packed = 0;
      rp.pred_aux = nullptr;
      rp.id_bits = 31;
      rp.id_mask = 0xFFFFFFFFu;
      rc = launch_rerank<unsigned long long, false>(ctx, cur, m, N, rp, ep, pool.p[2 * (cur ^ 1)], pool.p[2 * (cur ^ 1) + 1]);
      if (rc) return rc;
      S.algorithmic_bytes += (uint64_t)m * 12 + (uint64_t)m * 4;
    }
    h_next = std::min<uint64_t>((uint64_t)h32 * 2, 0x7FFFFFFFull);
    lean = !dbg && H.maxgroup > LEAN_MAXGROUP;  // (group sizes before this round; they rarely drop 8x in one)
    k_commit_sort<<<1, 1, 0, st>>>(ctx->d_state, ctx->d_ctrl(), (uint32_t)h_next, sel_of(cur), expect_cursor, lean ? 0u : 1u,
                                   0xFFFFFFFFu);
    CK(ctx, cudaGetLastError());
    S.kernel_launches++;
    if (r < BWTC_CUDA_MAX_ROUNDS) {
      S.live[r] = m;
      S.passes[r] = pdone;
      S.prefix_len[r] = h32;
      S.rounds = r + 1;
    }
    m_prev = m;
    ctx->last_cur = cur;
    lists_pending = true;
  }

  // ---- run statistics first: the verification below reuses d_scat
  if (finished && J.runs && !bs && J.block_mode) {
    S.algorithmic_bytes += 2ull * n;  // the run kernels read the output twice, once per block whatever the chunk count
    const uint32_t cnt = ctx->h_state->nruns;
    if (cnt <= J.runs->capacity && cnt <= n && J.runs->symbol && J.runs->start) {
      if (download_staged(ctx, J.runs->symbol, ctx->d_aux[0], cnt)) return BWTC_CUDA_ECUDA;
      if (download_staged(ctx, reinterpret_cast<uint8_t*>(J.runs->start), reinterpret_cast<const uint8_t*>(ctx->d_scat), (size_t)cnt * 4))
        return BWTC_CUDA_ECUDA;
      J.runs->count = cnt;
    } else {
      J.runs->count = BWTC_CUDA_RUNS_OVERFLOW;
    }
  }
  if (finished && verify) {
    rc = J.sa ? verify_sa(ctx, J) : verify_forward(ctx, J);
    if (rc) return rc;
  }
  // ---- result copies that could not be enqueued speculatively
  if (finished) {
    if (J.sa) {
      // the suffix array (its BWT bytes stay on the device): 4 bytes per suffix, direct from pinned memory, else staged
      if (J.h_sa && is_pinned_host(J.h_sa)) {
        CK(ctx, cudaMemcpyAsync(J.h_sa, J.sa, (size_t)N * 4, cudaMemcpyDeviceToHost, st));
        if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
      } else if (J.h_sa && download_staged(ctx, reinterpret_cast<uint8_t*>(J.h_sa), reinterpret_cast<const uint8_t*>(J.sa), (size_t)N * 4)) {
        return BWTC_CUDA_ECUDA;
      }
    } else if (bs) {
      if (!out_enqueued || !direct_out) {
        if (direct_out) {
          if (enqueue_direct_out() || host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
        } else {
          for (uint32_t k = 0; k < bs->nblocks; ++k) {
            const uint32_t nk = (k + 1 == bs->nblocks) ? bs->n_last : bs->n0;
            if (download_staged(ctx, static_cast<uint8_t*>(bs->out[k]), ctx->d_out + (size_t)k * J.bstride, nk)) return BWTC_CUDA_ECUDA;
          }
        }
      }
    } else if (!J.out_dev) {
      if (!J.block_mode) {
        // raw contract: U[pidx] stays untouched (divsufsort.c:506-512) — two ranges around it
        const uint32_t pidx = ctx->h_LF()[0];
        if (is_pinned_host(J.h_out)) {
          if (pidx > 0) CK(ctx, cudaMemcpyAsync(J.h_out, ctx->d_out, pidx, cudaMemcpyDeviceToHost, st));
          if (pidx + 1 < n) CK(ctx, cudaMemcpyAsync(J.h_out + pidx + 1, ctx->d_out + pidx + 1, n - pidx - 1, cudaMemcpyDeviceToHost, st));
          if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
        } else {
          if (download_staged(ctx, J.h_out, ctx->d_out, pidx)) return BWTC_CUDA_ECUDA;
          if (pidx + 1 < n && download_staged(ctx, J.h_out + pidx + 1, ctx->d_out + pidx + 1, n - pidx - 1)) return BWTC_CUDA_ECUDA;
        }
      } else if (!out_enqueued) {
        if (direct_out) {
          if (enqueue_direct_out() || host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
        } else if (download_staged(ctx, J.h_out, ctx->d_out, n)) {
          return BWTC_CUDA_ECUDA;
        }
      }
    }
  }
  // ---- results for the caller: LFpowers, freqs (incremented only now that the block has succeeded)
  if (bs) {
    const uint32_t* h_bhist = reinterpret_cast<const uint32_t*>(ctx->h_batch + MAX_BATCH * sizeof(void*));
    for (uint32_t k = 0; k < bs->nblocks; ++k) {
      const uint32_t nl = (k + 1 == bs->nblocks) ? bs->nLF_last : bs->nLF;
      for (uint32_t j = 0; j < nl; ++j) J.LF[k * 256 + j] = h_bLF[k * 256 + j];
      if (J.freqs)
        for (int c = 0; c < 256; ++c) J.freqs[k * 256 + c] += h_bhist[k * 256 + c];
    }
  } else {
    for (uint32_t j = 0; j < J.nLF; ++j) J.LF[j] = ctx->h_LF()[j];
    if (J.freqs)
      for (int c = 0; c < 256; ++c) J.freqs[c] += ctx->h_hist()[c];
  }
  float ms = 0;
  CK(ctx, cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end));
  S.gpu_ms = ms;
  if (ctx->timing_detail) {
    float tot = 0, tot0 = 0;
    for (size_t i = 0; i + 1 < pt.used; i += 2) {
      float t = 0;
      CK(ctx, cudaEventElapsedTime(&t, ctx->ev_pool[i], ctx->ev_pool[i + 1]));
      tot += t;
      if (i < round0_events) tot0 += t;
    }
    S.sort_ms = tot;
    S.sort0_ms = tot0;
  }
  return (int64_t)J.LF[0];
}

// Phase A, phase B, and the fallback of the static tile ids (see k_radix_pass): if the look-back watchdog fired, the
// context switches to ticket counters for good and repeats phase B.  The reversed, sentinel-terminated text is still
// intact on the device, so this works for in-place device buffers too; nothing was written to LFpowers / freqs.
int64_t run_job(bwtc_cuda_ctx* ctx, Job& J) {
  int64_t rc = phase_input(ctx, J);
  if (rc < 0) return rc;
  rc = phase_sort(ctx, J);
  if (rc == BWTC_CUDA_EINTERNAL && ctx->lb_watchdog && ctx->static_tiles) {
    ctx->static_tiles = 0;
    rc = phase_sort(ctx, J);
  }
  return rc;
}

int64_t run_transform(bwtc_cuda_ctx* ctx, bool block_mode, const uint8_t* h_in, uint8_t* h_out, const uint8_t* in_dev,
                      uint8_t* out_dev, uint32_t n, uint32_t* LF, uint32_t nLF, uint32_t* freqs,
                      const BatchSpec* bs = nullptr, bwtc_cuda_runs* runs = nullptr) {
  Job J;
  J.runs = runs;
  if (runs) runs->count = BWTC_CUDA_RUNS_OVERFLOW;
  J.block_mode = block_mode;
  J.h_in = h_in;
  J.h_out = h_out;
  J.in_dev = in_dev;
  J.out_dev = out_dev;
  J.n = n;
  J.LF = LF;
  J.nLF = nLF;
  J.freqs = freqs;
  J.bs = bs;
  const int64_t rc = run_job(ctx, J);
  // a failure after the runs were downloaded (EVERIFY, or an error in a later copy) must not leave a valid-looking count
  if (rc < 0 && runs) runs->count = BWTC_CUDA_RUNS_OVERFLOW;
  return rc;
}

// ---- inverse transform (SURVEY.md §8f row f4; kernels in ibwt_kernels.cuh).  block_mode: the n bytes a forward
// bwtc_cuda_bwt_block produced (hole at eob filled with L[N-1]), result n bytes of the original block — the contract of
// InverseBWTransform::doTransform(BWTBlock&) (InverseBWT.cpp:47-51).  raw: N = n_in bytes L[0..N) with L[eob] ignored,
// result N-1 bytes — the virtual doTransform(byte*, uint32, LFpow) (InverseBWT.hpp:49-50).
// The device part of an inversion (one block, or a batch of them, ibwt_kernels.cuh InvShape): ev_begin, the keys and C
// tables, the 2 digit passes, walk1, pointer jumping, walk2 into d_dst.  Adds its launches and algorithmic bytes to
// ctx->stats; nothing is waited for.  A batch (bhist != nullptr) counts per-block histograms and gets per-block C tables.
// Bit k of ctrl[CTR_INV_BAD..] ends up set for each block k that is not the BWT of any text.  verify (the verification of
// a forward transform): the walk kernels' VERIFY variants, which also check the LFpowers rows at sh.d_eob and honour
// sh.eot; ev_begin / ev_end are then left to the caller.
int enqueue_inverse(bwtc_cuda_ctx* ctx, const InvShape& sh, bool block_mode, const uint8_t* d_src, uint8_t* d_dst,
                    uint32_t* rounds_out, uint32_t* passes_out, bool verify = false) {
  const bool timed = !verify;
  cudaStream_t st = ctx->stream;
  bwtc_cuda_stats& S = ctx->stats;
  PassTimer pt{ctx};
  const uint32_t B = sh.nblocks, N = inv_rows(sh);
  uint32_t* bhist = B > 1 ? ctx->d_bhist : nullptr;
  if (timed) CK(ctx, cudaEventRecord(ctx->ev_begin, st));
  CK(ctx, cudaMemsetAsync(ctx->d_zero, 0, (size_t)CTR_STICKY * 4, st));
  if (zero_round_state(ctx, N, N, RS_TILE32, 3u)) return BWTC_CUDA_ECUDA;
  if (bhist) CK(ctx, cudaMemsetAsync(bhist, 0, (size_t)B * 256 * 4, st));
  uint32_t* keys0 = static_cast<uint32_t*>(ctx->d_keys[0]);
  uint32_t* C = ctx->d_ktab;  // B x 258 words (the lazy-rank prefix table is idle outside a forward transform)
  const dim3 kgrid(std::max<uint32_t>(1u, div_up((uint32_t)ctx->sm_count * 8u, B)), B);
  k_inv_keys<<<kgrid, 256, 0, st>>>(d_src, sh, block_mode ? 1 : 0, keys0, ctx->d_hist(), bhist);
  k_inv_ctable<<<B, 32, 0, st>>>(ctx->d_hist(), bhist, sh, C);
  CK(ctx, cudaGetLastError());
  S.kernel_launches += 2;
  S.algorithmic_bytes += (uint64_t)N * 5;
  int cur = 0;
  uint32_t pdone = 0;
  const int rc = run_sort<uint32_t, RS_IPT32>(ctx, N, 3u, true, N - 1, &cur, &pt, &pdone);
  if (rc) return rc;
  if (ctx->debug_fake_watchdog && ctx->static_tiles) {
    // test hook: the state a look-back watchdog in the digit passes leaves (every later kernel returns at entry)
    CK(ctx, cudaMemsetAsync(ctx->d_ctrl() + CTR_ERR, 0xFF, 4, st));
  }
  const uint32_t* vals = ctx->d_idx[cur];
  const uint32_t Sn = inv_splitters(sh);  // <= N / INV_K + B
  uint32_t* nxtA = ctx->d_scat;
  uint32_t* distA = nxtA + Sn;
  uint32_t* nxtB = distA + Sn;
  uint32_t* distB = nxtB + Sn;
  uint32_t* len = distB + Sn;  // 5 * ceil(N / INV_K) words fit d_scat (N + 16 words) unless N is tiny
  if ((uint64_t)5 * Sn > (uint64_t)N + 16) {  // tiny N: use the (idle) second id / key buffers as well (Sn <= N / 2)
    nxtA = ctx->d_idx[cur ^ 1]; distA = nxtA + Sn; nxtB = ctx->d_scat; distB = nxtB + Sn; len = static_cast<uint32_t*>(ctx->d_keys[1]);
  }
  const dim3 wgrid(div_up(sh.S0, 256), B);
  if (verify) k_inv_walk1<true><<<wgrid, 256, 0, st>>>(vals, sh, C, nxtA, len, ctx->d_ctrl());
  else k_inv_walk1<false><<<wgrid, 256, 0, st>>>(vals, sh, C, nxtA, len, ctx->d_ctrl());
  CK(ctx, cudaMemcpyAsync(distA, len, (size_t)Sn * 4, cudaMemcpyDeviceToDevice, st));
  uint32_t* nin = nxtA; uint32_t* din = distA; uint32_t* nout = nxtB; uint32_t* dout = distB;
  uint32_t rounds = 0;
  for (uint64_t span = 1; span < (uint64_t)sh.S0; span <<= 1) {  // a chain never leaves its block: ceil(log2 S0) rounds
    k_inv_jump<<<div_up(Sn, 256), 256, 0, st>>>(nin, din, Sn, nout, dout, ctx->d_ctrl());
    std::swap(nin, nout);
    std::swap(din, dout);
    ++rounds;
  }
  // single-cycle check: per-block length sums and CTA counters in the gram histogram words (zeroed above, idle here)
  if (verify) k_inv_walk2<true><<<wgrid, 256, 0, st>>>(vals, len, din, nin, C, sh, d_dst, ctx->d_ctrl(), ctx->d_hist() + GRAM_OFF);
  else k_inv_walk2<false><<<wgrid, 256, 0, st>>>(vals, len, din, nin, C, sh, d_dst, ctx->d_ctrl(), ctx->d_hist() + GRAM_OFF);
  CK(ctx, cudaGetLastError());
  S.kernel_launches += 2 + rounds;
  S.algorithmic_bytes += (uint64_t)N * (4 + 4 + 1) + (uint64_t)Sn * (16 * (rounds + 1) + 4);
  if (timed) CK(ctx, cudaEventRecord(ctx->ev_end, st));
  *rounds_out = rounds;
  *passes_out = pdone;
  return 0;
}

// spec (the single-block entry points): pinned host and device outputs are written without waiting for the check, so a
// valid block costs one host wait; a corrupt one leaves them unspecified.  !spec (a block of bwtc_cuda_inverse_blocks):
// restored into d_out, copied to the caller only if valid.  After a look-back watchdog the device part is repeated with
// ticket tile ids from the device copy of the input (d_in, or in_dev, which walk2 left untouched) — never from h_in, which
// the speculative copy may already have overwritten with stale bytes when it aliases a pinned h_out.
int64_t run_inverse(bwtc_cuda_ctx* ctx, bool block_mode, const uint8_t* h_in, uint8_t* h_out, const uint8_t* in_dev, uint8_t* out_dev,
                    uint32_t n_in, uint32_t eob, bool spec = true) {
  ctx->err[0] = 0;
  if (cudaSetDevice(ctx->device) != cudaSuccess) {
    set_err(ctx->err, "cudaSetDevice(%d) failed", ctx->device);
    return BWTC_CUDA_ECUDA;
  }
  const uint32_t N = block_mode ? n_in + 1u : n_in, n = N - 1u;
  if (n_in == 0 || n > ctx->cap || N < 2) {
    set_err(ctx->err, "inverse: block of %u bytes exceeds context capacity %u (or is empty)", n, ctx->cap);
    return n > ctx->cap ? BWTC_CUDA_ETOOBIG : BWTC_CUDA_EARG;
  }
  if (eob >= N) {
    set_err(ctx->err, "inverse: end-of-block position %u outside [0, %u)", eob, N);
    return BWTC_CUDA_EARG;
  }
  cudaStream_t st = ctx->stream;
  bwtc_cuda_stats& S = ctx->stats;
  const uint8_t* d_src = in_dev;
  if (!in_dev) {
    if (upload(ctx, ctx->d_in, h_in, n_in)) return BWTC_CUDA_ECUDA;
    d_src = ctx->d_in;
  }
  uint8_t* d_dst = (out_dev && spec) ? out_dev : ctx->d_out;
  const bool pinned_out = !out_dev && is_pinned_host(h_out);
  InvShape sh;
  sh.nblocks = 1;
  sh.R = sh.N_last = N;
  sh.n0 = sh.istride = n;
  sh.S0 = sh.S_last = div_up(N, INV_K);
  sh.eob[0] = eob;
  sh.d_eob = nullptr;
  uint32_t rounds = 0, pdone = 0;
  for (;;) {
    memset(&S, 0, sizeof(S));
    S.n_suffixes = N;
    S.batch_blocks = 1;
    if (const int rc = enqueue_inverse(ctx, sh, block_mode, d_src, d_dst, &rounds, &pdone)) return rc;
    CK(ctx, cudaMemcpyAsync(ctx->h_ctrl(), ctx->d_ctrl(), CTR_STICKY * 4, cudaMemcpyDeviceToHost, st));
    if (pinned_out && spec) CK(ctx, cudaMemcpyAsync(h_out, ctx->d_out, n, cudaMemcpyDeviceToHost, st));
    if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
    if (!ctx->h_ctrl()[CTR_ERR]) break;
    // the only look-back kernels here are the two digit passes; repeat with tickets (cannot happen twice)
    if (!ctx->static_tiles) {
      set_err(ctx->err, "inverse: look-back watchdog fired");
      return BWTC_CUDA_EINTERNAL;
    }
    ctx->static_tiles = 0;
  }
  const bool corrupt = (ctx->h_ctrl()[CTR_INV_BAD] & 1u) != 0u;
  if (!corrupt) {
    if (!spec && (out_dev || pinned_out)) {
      CK(ctx, cudaMemcpyAsync(out_dev ? out_dev : h_out, ctx->d_out, n, out_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
      if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
    } else if (!out_dev && !pinned_out && download_staged(ctx, h_out, ctx->d_out, n)) {
      return BWTC_CUDA_ECUDA;
    }
  }
  float ms = 0;
  CK(ctx, cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end));
  S.gpu_ms = ms;
  S.rounds = rounds;
  S.passes[0] = pdone;
  S.live[0] = N;
  S.flags = (ctx->static_tiles ? 0u : 1u) | (corrupt ? 128u : 0u);
  if (corrupt) {
    set_err(ctx->err, "inverse: block 0 is not the BWT of any text (with end-of-block row %u)", eob);
    return BWTC_CUDA_ECORRUPT;
  }
  return (int64_t)n;
}

// Verification of a finished forward transform (DESIGN.md §3.10): its device-resident output (J.d_dst, a batch at stride
// n0 + 1) is inverted into d_aux[1] — end-of-block rows read from d_LF on the device, every LFpowers entry checked against
// the rows the walk visits — and compared with the input, which d_text still holds reversed (block contract) or as it is
// (raw: T itself, whose restored N-1 bytes walk 2 writes reversed).  A raw text is one block whose end-of-text row has the
// key c = T[N-1] (ibwt_kernels.cuh k_inv_keys).  One host wait.  On failure an in-place device block is rewritten from
// d_text and BWTC_CUDA_EVERIFY is returned; nothing else of the caller's has been written yet.
int verify_forward(bwtc_cuda_ctx* ctx, const Job& J) {
  cudaStream_t st = ctx->stream;
  bwtc_cuda_stats& S = ctx->stats;
  const BatchSpec* bs = J.bs;
  InvShape sh;
  sh.nblocks = bs ? bs->nblocks : 1u;
  sh.n0 = bs ? bs->n0 : J.n;
  sh.istride = bs ? J.bstride : J.n;
  sh.R = bs ? J.bstride : J.N;
  sh.N_last = bs ? bs->n_last + 1u : J.N;
  sh.S0 = div_up(sh.R, INV_K);
  sh.S_last = div_up(sh.N_last, INV_K);
  sh.d_eob = ctx->d_LF;
  sh.eot[0] = J.block_mode ? 0 : J.last;
  sh.nLF = J.nLF;
  sh.nLF_last = bs ? bs->nLF_last : J.nLF;
  if (ctx->debug_corrupt_out) {
    if (J.block_mode) k_debug_flip_byte<<<1, 1, 0, st>>>(J.d_dst + sh.n0 / 2);
    else k_debug_flip_raw<<<1, 1, 0, st>>>(J.d_dst, J.N / 2, J.N, ctx->d_LF);
    CK(ctx, cudaGetLastError());
    S.kernel_launches++;
  }
  if (ctx->debug_corrupt_lf) {
    k_debug_corrupt_lf<<<1, MAX_BATCH, 0, st>>>(ctx->d_LF, ctx->debug_corrupt_lf, sh.nblocks, sh.nLF, sh.nLF_last);
    CK(ctx, cudaGetLastError());
    S.kernel_launches++;
  }
  for (;;) {
    uint32_t rounds = 0, pdone = 0;
    if (const int rc = enqueue_inverse(ctx, sh, J.block_mode, J.d_dst, ctx->d_aux[1], &rounds, &pdone, true)) return rc;
    const dim3 vgrid(std::max<uint32_t>(1u, div_up((uint32_t)ctx->sm_count * 8u, sh.nblocks)), sh.nblocks);
    k_inv_verify<<<vgrid, 256, 0, st>>>(ctx->d_aux[1], J.d_text, sh, ctx->d_ctrl());
    CK(ctx, cudaGetLastError());
    S.kernel_launches++;
    S.algorithmic_bytes += 2ull * J.n;
    CK(ctx, cudaEventRecord(ctx->ev_end, st));
    CK(ctx, cudaMemcpyAsync(ctx->h_ctrl(), ctx->d_ctrl(), CTR_STICKY * 4, cudaMemcpyDeviceToHost, st));
    if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
    if (!ctx->h_ctrl()[CTR_ERR]) break;
    if (!ctx->static_tiles) {
      set_err(ctx->err, "verification: look-back watchdog fired in the inverse");
      return BWTC_CUDA_EINTERNAL;
    }
    ctx->static_tiles = 0;  // the inverse's two digit passes again with ticket tile ids (cannot fire twice)
  }
  S.flags |= 64u;
  const uint64_t mask = (uint64_t)ctx->h_ctrl()[CTR_INV_BAD] | ((uint64_t)ctx->h_ctrl()[CTR_INV_BAD + 1] << 32);
  if (!mask) return 0;
  if (!bs && J.block_mode && J.out_dev && J.out_dev == J.in_dev) {
    k_text_unreverse<<<ctx->sm_count * 4, 256, 0, st>>>(J.d_text, J.n, J.out_dev);
    CK(ctx, cudaGetLastError());
    S.kernel_launches++;
    if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
  }
  uint32_t first = 0;
  while (!((mask >> first) & 1u)) ++first;
  set_err(ctx->err, "verification failed: the forward output of block %u of %u does not restore its input", first, sh.nblocks);
  return BWTC_CUDA_EVERIFY;
}

// sufcheck on the device (bwt_kernels.cuh k_sa_perm / k_sa_order): ISA in d_keys[0], idle outside a transform.  Enqueues
// the check and the read-back of the control words into h_ctrl; the caller waits.
int enqueue_sufcheck(bwtc_cuda_ctx* ctx, const uint8_t* d_text, const int32_t* d_sa, uint32_t n) {
  cudaStream_t st = ctx->stream;
  uint32_t* isa = static_cast<uint32_t*>(ctx->d_keys[0]);
  CK(ctx, cudaMemsetAsync(ctx->d_ctrl() + CTR_SA_BAD, 0, 8, st));
  CK(ctx, cudaMemsetAsync(isa, 0xFF, (size_t)n * 4, st));
  const uint32_t grid = std::max<uint32_t>(1u, std::min<uint32_t>(div_up(n, 256), (uint32_t)ctx->sm_count * 8u));
  k_sa_perm<<<grid, 256, 0, st>>>(d_sa, n, isa, ctx->d_ctrl());
  k_sa_order<<<grid, 256, 0, st>>>(d_text, d_sa, n, isa, ctx->d_ctrl());
  CK(ctx, cudaGetLastError());
  CK(ctx, cudaMemcpyAsync(ctx->h_ctrl(), ctx->d_ctrl(), CTR_STICKY * 4, cudaMemcpyDeviceToHost, st));
  ctx->stats.kernel_launches += 2;
  ctx->stats.algorithmic_bytes += (uint64_t)n * 4 * 4 + (uint64_t)n * 13;  // ISA fill + SA twice + ISA min; 3 ISA / 1 T gathers
  return 0;
}

// After the wait: 0 if the check passed, else 1 with the first failing row and its reason in ctx->err.
int sufcheck_failed(bwtc_cuda_ctx* ctx, uint32_t n, const char* what) {
  const uint64_t w = (uint64_t)ctx->h_ctrl()[CTR_SA_BAD] | ((uint64_t)ctx->h_ctrl()[CTR_SA_BAD + 1] << 32);
  if (!w) return 0;
  const uint64_t key = ~w;
  const uint32_t row = (uint32_t)((key >> 2) & 0xFFFFFFFFull), reason = (uint32_t)(key & 3u);
  set_err(ctx->err, "%s: row %u of %u: %s", what, row, n,
          reason == SA_BAD_RANGE ? "value out of range" :
          reason == SA_BAD_DUP ? "duplicate (an earlier row holds the same value)" :
          "out of order (its suffix does not sort after the one of the row before)");
  return 1;
}

// Verification of a suffix array (bwtc_cuda_divsufsort with verification on, DESIGN.md §3.11): sufcheck on the device
// against the text it was sorted from, before anything is copied to the caller.  One host wait.
int verify_sa(bwtc_cuda_ctx* ctx, const Job& J) {
  cudaStream_t st = ctx->stream;
  bwtc_cuda_stats& S = ctx->stats;
  if (ctx->debug_corrupt_sa >= 0 && (uint64_t)ctx->debug_corrupt_sa + 1 < J.N) {
    k_debug_swap_sa<<<1, 1, 0, st>>>(J.sa, (uint32_t)ctx->debug_corrupt_sa);
    CK(ctx, cudaGetLastError());
    S.kernel_launches++;
  }
  if (enqueue_sufcheck(ctx, J.d_text, J.sa, J.N)) return BWTC_CUDA_ECUDA;
  CK(ctx, cudaEventRecord(ctx->ev_end, st));
  if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
  S.flags |= 64u;
  return sufcheck_failed(ctx, J.N, "verification failed: the suffix array") ? BWTC_CUDA_EVERIFY : 0;
}

// bwtc_cuda_divsufsort(_device): the raw transform with SA emission into d_sa; h_sa receives a copy.
int run_divsufsort(bwtc_cuda_ctx* ctx, const uint8_t* h_T, const uint8_t* d_T, int32_t* h_SA, int32_t* d_SA, uint32_t n) {
  uint32_t pidx = 0;
  Job J;
  J.block_mode = false;
  J.h_in = h_T;
  J.in_dev = d_T;
  J.n = n;
  J.LF = &pidx;
  J.nLF = 1;
  J.sa = d_SA;
  J.h_sa = h_SA;
  const int64_t rc = run_job(ctx, J);
  return rc < 0 ? (int)rc : 0;
}

// count blocks (block contract) through one context: as ONE batch when they qualify — 2..MAX_BATCH blocks, all of
// sizes[0] bytes except the last which may be shorter, together within the context's capacity, and at least one byte
// value unused (the batch reserves a code for its sentinels) — otherwise one after the other.  Results are
// identical either way.  LF = [count][256], nLF = [count], freqs = [count][256] or nullptr.
bool batchable(const bwtc_cuda_ctx* ctx, const uint32_t* sizes, uint32_t count) {
  if (!ctx->use_batch || count < 2 || count > MAX_BATCH) return false;
  uint64_t total = 0;
  for (uint32_t k = 0; k < count; ++k) {
    if (sizes[k] == 0) return false;
    if (k + 1 < count ? sizes[k] != sizes[0] : sizes[k] > sizes[0]) return false;
    total += (uint64_t)sizes[k] + 1;
  }
  return total <= (uint64_t)ctx->cap + 1 && total <= (uint64_t)BWTC_CUDA_MAX_BLOCK;
}

int transform_batch(bwtc_cuda_ctx* ctx, const void* const* in, void* const* out, const uint32_t* sizes, uint32_t count,
                    uint32_t starts, bool on_device, uint32_t* LF, uint32_t* nLF, uint32_t* freqs, bwtc_cuda_stats* stats,
                    bwtc_cuda_runs* runs = nullptr /* count == 1, host block only */) {
  for (uint32_t k = 0; k < count; ++k) {
    if (!in[k] || !out[k] || sizes[k] == 0) { set_err(ctx->err, "null or empty block %u", k); return BWTC_CUDA_EARG; }
    nLF[k] = bwtc_cuda_num_starting_points(sizes[k], starts);
  }
  if (batchable(ctx, sizes, count)) {
    BatchSpec bs;
    bs.nblocks = count;
    bs.n0 = sizes[0];
    bs.n_last = sizes[count - 1];
    bs.in = in;
    bs.out = out;
    bs.on_device = on_device;
    bs.LF = LF;
    bs.nLF = nLF[0];
    bs.nLF_last = nLF[count - 1];
    bs.freqs = freqs;
    const int64_t rc = run_transform(ctx, true, nullptr, nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, &bs);
    if (rc != BATCH_NEEDS_SINGLE) {
      ctx->stats.batch_blocks = count;  // the record describes the whole batch: count it once, not per block
      if (stats) for (uint32_t k = 0; k < count; ++k) stats[k] = ctx->stats;
      return rc < 0 ? (int)rc : 0;
    }
  }
  for (uint32_t k = 0; k < count; ++k) {
    uint32_t* fr = freqs ? freqs + (size_t)k * 256 : nullptr;
    int64_t rc;
    if (on_device)
      rc = run_transform(ctx, true, nullptr, nullptr, static_cast<const uint8_t*>(in[k]), static_cast<uint8_t*>(out[k]), sizes[k],
                         LF + (size_t)k * 256, nLF[k], fr);
    else
      rc = run_transform(ctx, true, static_cast<const uint8_t*>(in[k]), static_cast<uint8_t*>(out[k]), nullptr, nullptr, sizes[k],
                         LF + (size_t)k * 256, nLF[k], fr, nullptr, count == 1 ? runs : nullptr);
    ctx->stats.batch_blocks = 1;
    if (stats) stats[k] = ctx->stats;
    if (rc < 0) return (int)rc;
  }
  return 0;
}

// 2..MAX_BATCH blocks (block contract) that batchable() accepts, inverted as ONE device-side problem (DESIGN.md §3.7).  The
// caller has checked the arguments.  The blocks are staged in d_in (stride n0) and restored into d_out; the caller's
// buffers are written only after the host has read CTR_ERR.  After a look-back watchdog the device part is repeated with
// ticket tile ids from the staged input — never from the caller's buffers, which may alias the outputs.
// *bad: bit k set = block k is corrupt; its buffer is not written, and the call returns BWTC_CUDA_ECORRUPT.
int run_inverse_batch(bwtc_cuda_ctx* ctx, const void* const* in, void* const* out, const uint32_t* sizes, uint32_t count,
                      bool on_device, const uint32_t* eobs, uint64_t* bad) {
  *bad = 0;
  ctx->err[0] = 0;
  if (cudaSetDevice(ctx->device) != cudaSuccess) {
    set_err(ctx->err, "cudaSetDevice(%d) failed", ctx->device);
    return BWTC_CUDA_ECUDA;
  }
  static_assert(INV_MAX_BLOCKS == MAX_BATCH, "InvShape holds one end-of-block row per block of a batch");
  cudaStream_t st = ctx->stream;
  InvShape sh;
  sh.nblocks = count;
  sh.n0 = sh.istride = sizes[0];
  sh.R = sizes[0] + 1u;
  sh.d_eob = nullptr;
  sh.N_last = sizes[count - 1] + 1u;
  sh.S0 = div_up(sh.R, INV_K);
  sh.S_last = div_up(sh.N_last, INV_K);
  for (uint32_t k = 0; k < count; ++k) sh.eob[k] = eobs[k];
  for (uint32_t k = 0; k < count; ++k) {
    uint8_t* d = ctx->d_in + (size_t)k * sh.n0;
    if (on_device) CK(ctx, cudaMemcpyAsync(d, in[k], sizes[k], cudaMemcpyDeviceToDevice, st));
    else if (upload(ctx, d, static_cast<const uint8_t*>(in[k]), sizes[k])) return BWTC_CUDA_ECUDA;
  }
  bwtc_cuda_stats& S = ctx->stats;
  uint32_t rounds = 0, pdone = 0;
  for (;;) {
    memset(&S, 0, sizeof(S));
    if (const int rc = enqueue_inverse(ctx, sh, true, ctx->d_in, ctx->d_out, &rounds, &pdone)) return rc;
    CK(ctx, cudaMemcpyAsync(ctx->h_ctrl(), ctx->d_ctrl(), CTR_STICKY * 4, cudaMemcpyDeviceToHost, st));
    if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
    if (!ctx->h_ctrl()[CTR_ERR]) break;
    if (!ctx->static_tiles) {
      set_err(ctx->err, "inverse: look-back watchdog fired");
      return BWTC_CUDA_EINTERNAL;
    }
    ctx->static_tiles = 0;  // the two digit passes again with ticket tile ids (cannot fire twice)
  }
  const uint64_t mask = (uint64_t)ctx->h_ctrl()[CTR_INV_BAD] | ((uint64_t)ctx->h_ctrl()[CTR_INV_BAD + 1] << 32);
  bool pending = false;
  for (uint32_t k = 0; k < count; ++k) {
    if ((mask >> k) & 1u) continue;  // a corrupt block's buffer stays as it was
    const uint8_t* d = ctx->d_out + (size_t)k * sh.n0;
    uint8_t* o = static_cast<uint8_t*>(out[k]);
    if (on_device) {
      CK(ctx, cudaMemcpyAsync(o, d, sizes[k], cudaMemcpyDeviceToDevice, st));
      pending = true;
    } else if (is_pinned_host(o)) {
      CK(ctx, cudaMemcpyAsync(o, d, sizes[k], cudaMemcpyDeviceToHost, st));
      pending = true;
    } else if (download_staged(ctx, o, d, sizes[k])) {
      return BWTC_CUDA_ECUDA;
    }
  }
  if (pending && host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
  float ms = 0;
  CK(ctx, cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end));
  S.n_suffixes = inv_rows(sh);
  S.batch_blocks = count;
  S.gpu_ms = ms;
  S.rounds = rounds;
  S.passes[0] = pdone;
  S.live[0] = S.n_suffixes;
  S.flags = 2u | (ctx->static_tiles ? 0u : 1u);
  *bad = mask;
  return mask ? BWTC_CUDA_ECORRUPT : 0;
}

// count blocks (block contract) through one context, each restored as run_inverse would: runs are formed greedily as in
// bwtc_cuda_bwt_blocks, a run that batchable() accepts is inverted as one problem, any other block on its own.  Every
// argument is checked before any work, so a bad block leaves all caller buffers untouched.  stats: count records (the
// blocks of a batch share one) or nullptr.
int inverse_blocks(bwtc_cuda_ctx* ctx, const void* const* in, void* const* out, const uint32_t* sizes, uint32_t count,
                   bool on_device, const uint32_t* eobs, bwtc_cuda_stats* stats) {
  for (uint32_t k = 0; k < count; ++k) {
    if (!in[k] || !out[k] || sizes[k] == 0) { set_err(ctx->err, "inverse: null or empty block %u", k); return BWTC_CUDA_EARG; }
    if (sizes[k] > ctx->cap) {
      set_err(ctx->err, "inverse: block %u of %u bytes exceeds context capacity %u", k, sizes[k], ctx->cap);
      return BWTC_CUDA_ETOOBIG;
    }
    if (eobs[k] > sizes[k]) {
      set_err(ctx->err, "inverse: end-of-block position %u of block %u outside [0, %u)", eobs[k], k, sizes[k] + 1u);
      return BWTC_CUDA_EARG;
    }
  }
  uint32_t ncorrupt = 0, first_corrupt = 0;
  for (uint32_t k0 = 0; k0 < count;) {
    uint32_t k1 = std::min<uint32_t>(count, k0 + MAX_BATCH);
    while (k1 > k0 + 1 && !batchable(ctx, sizes + k0, k1 - k0)) --k1;
    int64_t rc;
    uint64_t bad = 0;
    if (k1 - k0 >= 2)
      rc = run_inverse_batch(ctx, in + k0, out + k0, sizes + k0, k1 - k0, on_device, eobs + k0, &bad);
    else if (on_device)
      rc = run_inverse(ctx, true, nullptr, nullptr, static_cast<const uint8_t*>(in[k0]), static_cast<uint8_t*>(out[k0]), sizes[k0],
                       eobs[k0], false);
    else
      rc = run_inverse(ctx, true, static_cast<const uint8_t*>(in[k0]), static_cast<uint8_t*>(out[k0]), nullptr, nullptr, sizes[k0],
                       eobs[k0], false);
    if (rc == BWTC_CUDA_ECORRUPT && k1 - k0 == 1) bad = 1u;
    else if (rc < 0 && rc != BWTC_CUDA_ECORRUPT) return (int)rc;
    for (uint32_t k = k0; k < k1; ++k) {
      const bool b = (bad >> (k - k0)) & 1u;
      if (b && !ncorrupt++) first_corrupt = k;
      if (stats) {
        stats[k] = ctx->stats;
        stats[k].flags = (ctx->stats.flags & ~128u) | (b ? 128u : 0u);
      }
    }
    k0 = k1;
  }
  if (ncorrupt) {
    set_err(ctx->err, "inverse: block %u (%u of %u blocks corrupt) is not the BWT of any text (with end-of-block row %u)",
            first_corrupt, ncorrupt, count, eobs[first_corrupt]);
    return BWTC_CUDA_ECORRUPT;
  }
  return 0;
}

}  // namespace

// =====================================================================================================
// extern "C"
// =====================================================================================================
extern "C" {

int bwtc_cuda_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    set_err(g_err, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    return BWTC_CUDA_ECUDA;
  }
  return n;
}

#define BWTC_STR2(x) #x
#define BWTC_STR(x) BWTC_STR2(x)
const char* bwtc_cuda_version(void) {
  return "bwtc_b200 0.1 sm_100a radix-pass BLOCK=" BWTC_STR(BWTC_RS_BLOCK) " IPT64=" BWTC_STR(BWTC_RS_IPT64)
         " IPT32=" BWTC_STR(BWTC_RS_IPT32);
}

const char* bwtc_cuda_global_error(void) { return g_err; }

uint32_t bwtc_cuda_stats_sizeof(void) { return (uint32_t)sizeof(bwtc_cuda_stats); }

int bwtc_cuda_ctx_create(bwtc_cuda_ctx** out, int device, uint32_t max_block_bytes) {
  if (!out || max_block_bytes == 0) { set_err(g_err, "bad arguments"); return BWTC_CUDA_EARG; }
  if (max_block_bytes > BWTC_CUDA_MAX_BLOCK) { set_err(g_err, "max_block_bytes above engine limit"); return BWTC_CUDA_ETOOBIG; }
  *out = nullptr;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) { set_err(g_err, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e)); return BWTC_CUDA_ECUDA; }
  bwtc_cuda_ctx* c = new (std::nothrow) bwtc_cuda_ctx();
  if (!c) { set_err(g_err, "out of host memory"); return BWTC_CUDA_EALLOC; }
  c->device = device;
  c->cap = max_block_bytes;
  if (const char* e = getenv("BWTC_STATIC_TILES")) c->static_tiles = atoi(e);
  if (const char* e = getenv("BWTC_DEBUG_FAKE_WATCHDOG")) c->debug_fake_watchdog = atoi(e);
  if (const char* e = getenv("BWTC_DEBUG_REVERSE_TILES")) c->debug_reverse_tiles = atoi(e);
  if (const char* e = getenv("BWTC_VERIFY")) c->verify = atoi(e) ? 1 : 0;
  if (const char* e = getenv("BWTC_DEBUG_CORRUPT_OUT")) c->debug_corrupt_out = atoi(e);
  if (const char* e = getenv("BWTC_DEBUG_CORRUPT_LF")) c->debug_corrupt_lf = (uint32_t)std::max(0, atoi(e));
  if (const char* e = getenv("BWTC_DEBUG_CORRUPT_SA")) c->debug_corrupt_sa = std::max(-1L, atol(e));
  if (const char* e = getenv("BWTC_DEBUG_SKIP_COPIES")) c->debug_skip_copies = atoi(e);
  if (const char* e = getenv("BWTC_D2H_KERNEL")) c->d2h_kernel = atoi(e);
  if (const char* e = getenv("BWTC_D2H_CTAS")) c->d2h_ctas = std::max(1, atoi(e));
  if (const char* e = getenv("BWTC_SPIN_WAIT")) c->wait_mode = atoi(e) ? 1 : 0;
  if (const char* e = getenv("BWTC_WAIT_MODE")) c->wait_mode = atoi(e);
  if (const char* e = getenv("BWTC_POLL_SPIN_US")) c->poll_spin_us = std::max(0, atoi(e));
  if (const char* e = getenv("BWTC_POLL_SLEEP_US")) c->poll_sleep_us = std::max(1, atoi(e));
  if (const char* e = getenv("BWTC_LADDER_FIRST")) c->ladder_first = std::max(0, atoi(e));
  if (const char* e = getenv("BWTC_LADDER_MORE")) c->ladder_more = std::max(1, atoi(e));
  if (const char* e = getenv("BWTC_LAZY")) c->use_lazy = atoi(e);
  if (const char* e = getenv("BWTC_HYBRID2")) c->hybrid2 = atoi(e);
  if (const char* e = getenv("BWTC_TWOPASS")) c->twopass = atoi(e);
  if (const char* e = getenv("BWTC_GRAM")) c->use_gram = atoi(e);
  if (const char* e = getenv("BWTC_PARTIAL")) c->use_partial = atoi(e);
  if (const char* e = getenv("BWTC_RERANK_PF")) c->rerank_pf_tiles = (uint32_t)std::max(0, atoi(e));
  c->use_radix9 = env_radix9();
  c->status_row_words = status_row_words_for(c->use_radix9);
  if (const char* e = getenv("BWTC_LAZY_MIN_MIB")) c->lazy_min_suffixes = (uint32_t)std::max(0L, atol(e)) << 20;
  if (const char* e = getenv("BWTC_LAZY_MAX_LIVE")) c->lazy_max_live = atof(e);
  if (const char* e = getenv("BWTC_LAZY_MAX_REPEATS")) c->lazy_max_repeats = atof(e);
  if (const char* e = getenv("BWTC_SEG")) c->use_seg = atoi(e);
  if (const char* e = getenv("BWTC_BATCH")) c->use_batch = atoi(e);
  if (const char* e = getenv("BWTC_PACK_PRED")) c->use_pack_pred = atoi(e);
  if (const char* e = getenv("BWTC_AUX_MIN_MIB")) { const long v = atol(e); c->aux_min_suffixes = v > 0 ? (uint32_t)v << 20 : (v == 0 ? 1u : 0u); }
  if (const char* e = getenv("BWTC_BUCKET_MIN_WINDOWS")) c->bucket_min_windows = atoi(e);
  if (const char* e = getenv("BWTC_RERANK_WINDOW_MB")) { long v = atol(e); if (v > 0) c->rerank_window_bytes = (uint64_t)v << 20; }
  c->err[0] = 0;
  memset(&c->stats, 0, sizeof(c->stats));
  const size_t N = (size_t)max_block_bytes + 1;
  const uint32_t min_tile = RS_TILE64 < RS_TILE32 ? RS_TILE64 : RS_TILE32;
  c->max_rs_tiles = div_up(N, min_tile);
  c->max_aux_tiles = div_up(N, AUX_TILE);
  int rc = 0;
#define ALLOC(ptr, bytes)                                                                       \
  do {                                                                                          \
    if (!rc) {                                                                                  \
      e = cudaMalloc((void**)&(ptr), (bytes));                                                  \
      if (e != cudaSuccess) {                                                                   \
        set_err(g_err, "cudaMalloc(%zu bytes) for " #ptr ": %s", (size_t)(bytes), cudaGetErrorString(e)); \
        rc = BWTC_CUDA_EALLOC;                                                                  \
      }                                                                                         \
    }                                                                                           \
  } while (0)
  int sm = 0;
  if (cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sm > 0) c->sm_count = sm;
  {  // refuse up front, with a clear message, what the device cannot hold (instead of failing half way through the list)
    size_t free_b = 0, total_b = 0;
    const uint64_t need = bwtc_cuda_scratch_bytes(max_block_bytes);
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && need > (uint64_t)free_b) {
      set_err(g_err, "a context for %u-byte blocks needs %llu bytes of device memory, %llu are free", max_block_bytes,
              (unsigned long long)need, (unsigned long long)free_b);
      delete c;
      return BWTC_CUDA_EALLOC;
    }
  }
  e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { set_err(g_err, "cudaStreamCreate: %s", cudaGetErrorString(e)); rc = BWTC_CUDA_ECUDA; }
  const size_t padded = ((N + TEXT_PAD + 15) / 16) * 16 + 16;
  ALLOC(c->d_in, padded);
  ALLOC(c->d_text, padded);
  ALLOC(c->d_out, padded);
  ALLOC(c->d_rank, (N + 64) * 4);
  ALLOC(c->d_keys[0], N * 8 + 64);  // (+ one sector: rank_lookup reads whole 32-byte sectors of the sorted keys)
  ALLOC(c->d_keys[1], N * 8 + 64);
  ALLOC(c->d_idx[0], N * 4);
  ALLOC(c->d_idx[1], N * 4);
  ALLOC(c->d_zero, (size_t)(CTR_WORDS + HIST_WORDS) * 4 + (size_t)MAX_RERANK_WINDOWS * c->max_aux_tiles * 8 + 64);
  ALLOC(c->d_status, (size_t)MAX_PASSES * (c->max_rs_tiles + LB_PAD_ROWS) * c->status_row_words * 4u);
  ALLOC(c->d_LF, (size_t)LF_WORDS * 4);
  ALLOC(c->d_state, sizeof(LadderState));
  ALLOC(c->d_livebits, (N / 32 + 4) * 4);
  ALLOC(c->d_ktab, ((size_t)(1u << KTAB_BITS) + 2) * 4);
  ALLOC(c->d_lookup, sizeof(LookupParams));
  ALLOC(c->d_bhist, (size_t)MAX_BATCH * 256 * 4);
  ALLOC(c->d_bptr, (size_t)MAX_BATCH * sizeof(void*));
  ALLOC(c->d_wtab, (size_t)WS_SLOTS * 12 + 64);
  ALLOC(c->d_tilecnt, (size_t)c->max_aux_tiles * (2 + MAX_RERANK_WINDOWS + 1) * 4 + 64);
  ALLOC(c->d_scat, (size_t)N * 4 + 64);
  ALLOC(c->d_aux[0], padded);
  ALLOC(c->d_aux[1], padded);
#undef ALLOC
  if (!rc) {  // pad rows of the look-back status: "inclusive prefix = 0", never overwritten
    std::vector<uint32_t> pad((size_t)LB_PAD_ROWS * c->status_row_words, LB_PAD_WORD);
    for (int p = 0; p < MAX_PASSES && !rc; ++p) {
      e = cudaMemcpy(status_rows(c, p) - pad.size(), pad.data(), pad.size() * 4, cudaMemcpyHostToDevice);
      if (e != cudaSuccess) { set_err(g_err, "cudaMemcpy(status pad): %s", cudaGetErrorString(e)); rc = BWTC_CUDA_ECUDA; }
    }
  }
  if (!rc) {
    e = cudaMallocHost((void**)&c->h_small, (size_t)(CTR_WORDS + HIST_WORDS + 256 + 8) * 4);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&c->h_batch, (size_t)MAX_BATCH * (sizeof(void*) + 2 * 256 * 4));
    if (e == cudaSuccess) e = cudaMallocHost((void**)&c->h_state, sizeof(LadderState));
    if (e == cudaSuccess) e = cudaMallocHost((void**)&c->h_lookup, sizeof(LookupParams));
    if (e != cudaSuccess) { set_err(g_err, "cudaMallocHost: %s", cudaGetErrorString(e)); rc = BWTC_CUDA_EALLOC; }
  }
  if (!rc && (cudaEventCreate(&c->ev_begin) != cudaSuccess || cudaEventCreate(&c->ev_end) != cudaSuccess ||
              cudaEventCreateWithFlags(&c->ev_sync, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess ||
              cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming) != cudaSuccess ||
              cudaEventCreateWithFlags(&c->ev_comp, cudaEventDisableTiming) != cudaSuccess)) {
    set_err(g_err, "cudaEventCreate failed");
    rc = BWTC_CUDA_ECUDA;
  }
  if (!rc) {
    if (const char* sl = getenv("BWTC_DEBUG_SPIN_LIMIT")) {  // test hook: a watchdog that fires within milliseconds
      const uint32_t v = (uint32_t)std::max(1L, atol(sl));
      if (cudaMemcpyToSymbol(g_lb_spin_limit, &v, sizeof(v)) != cudaSuccess) { set_err(g_err, "cudaMemcpyToSymbol failed"); rc = BWTC_CUDA_ECUDA; }
    }
  }
  if (!rc) {
    int r2 = 0;
    r2 |= set_pass_attr<uint32_t, RS_IPT32, true, false>(c);
    r2 |= set_pass_attr<uint32_t, RS_IPT32, false, false>(c);
    r2 |= set_pass_attr<unsigned long long, RS_IPT64, true, false>(c);
    r2 |= set_pass_attr<unsigned long long, RS_IPT64, false, false>(c);
    r2 |= set_pass_attr<uint32_t, RS_IPT32, true, true>(c);
    r2 |= set_pass_attr<uint32_t, RS_IPT32, false, true>(c);
    r2 |= set_pass_attr<unsigned long long, RS_IPT64, true, true>(c);
    r2 |= set_pass_attr<unsigned long long, RS_IPT64, false, true>(c);
    r2 |= set_pass_attr<unsigned long long, RS_IPT64, true, false, 9>(c);
    r2 |= set_pass_attr<unsigned long long, RS_IPT64, false, false, 9>(c);
    r2 |= set_pass_attr<unsigned long long, RS_IPT64, true, true, 9>(c);
    r2 |= set_pass_attr<unsigned long long, RS_IPT64, false, true, 9>(c);
    if (r2) { set_err(g_err, "%s", c->err); rc = BWTC_CUDA_ECUDA; }
  }
  if (rc) { ctx_free(c); return rc; }
#ifdef BWTC_PROFILE_STAGES
  {
    unsigned long long* pbuf = nullptr;
    cudaMalloc((void**)&pbuf, c->max_rs_tiles * 16 * 8);
    cudaMemset(pbuf, 0, c->max_rs_tiles * 16 * 8);
    cudaMemcpyToSymbol(g_prof_buf, &pbuf, sizeof(pbuf));
  }
#endif
  *out = c;
  return 0;
}

void bwtc_cuda_ctx_destroy(bwtc_cuda_ctx* ctx) { ctx_free(ctx); }

/* The device allocations of bwtc_cuda_ctx_create, summed (keep in step with its ALLOC list). */
uint64_t bwtc_cuda_scratch_bytes(uint32_t max_block_bytes) {
  const uint64_t N = (uint64_t)max_block_bytes + 1;
  const uint32_t min_tile = RS_TILE64 < RS_TILE32 ? RS_TILE64 : RS_TILE32;
  const uint64_t rs_tiles = div_up(N, min_tile), aux_tiles = div_up(N, AUX_TILE);
  const uint64_t padded = ((N + TEXT_PAD + 15) / 16) * 16 + 16;
  uint64_t b = 5 * padded;                                  // d_in, d_text, d_out, d_aux[2]
  b += (N + 64) * 4;                                        // d_rank
  b += 2 * (N * 8 + 64) + 2 * N * 4;                        // d_keys[2], d_idx[2]
  b += N * 4 + 64;                                          // d_scat
  b += (uint64_t)(CTR_WORDS + HIST_WORDS) * 4 + (uint64_t)MAX_RERANK_WINDOWS * aux_tiles * 8 + 64;  // d_zero
  b += (uint64_t)MAX_PASSES * (rs_tiles + LB_PAD_ROWS) * status_row_words_for(env_radix9()) * 4u;     // d_status
  b += (uint64_t)LF_WORDS * 4 + sizeof(LadderState) + (uint64_t)MAX_BATCH * 256 * 4 + (uint64_t)MAX_BATCH * sizeof(void*);
  b += (uint64_t)WS_SLOTS * 12 + 64;                        // d_wtab
  b += aux_tiles * (2 + MAX_RERANK_WINDOWS + 1) * 4 + 64;   // d_tilecnt
  b += (N / 32 + 4) * 4 + ((uint64_t)(1u << KTAB_BITS) + 2) * 4 + sizeof(LookupParams);  // lazy ranks: d_livebits, d_ktab, d_lookup
  return b;
}

const char* bwtc_cuda_last_error(const bwtc_cuda_ctx* ctx) { return ctx ? ctx->err : g_err; }

int bwtc_cuda_get_stats(const bwtc_cuda_ctx* ctx, bwtc_cuda_stats* out) {
  if (!ctx || !out) return BWTC_CUDA_EARG;
  *out = ctx->stats;
  return 0;
}

int bwtc_cuda_ctx_set_round0(bwtc_cuda_ctx* ctx, uint32_t chars, uint32_t key_bytes) {
  if (!ctx || (key_bytes != 0 && key_bytes != 4 && key_bytes != 8) || chars > 64) return BWTC_CUDA_EARG;
  ctx->force_chars = chars;
  ctx->force_keybytes = key_bytes;
  return 0;
}

int bwtc_cuda_ctx_set_timing(bwtc_cuda_ctx* ctx, int detail) {
  if (!ctx) return BWTC_CUDA_EARG;
  if (detail && ctx->ev_pool.empty()) {
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BWTC_CUDA_ECUDA;
    ctx->ev_pool.resize(2 * MAX_PASSES * BWTC_CUDA_MAX_ROUNDS);
    for (auto& ev : ctx->ev_pool)
      if (cudaEventCreate(&ev) != cudaSuccess) { set_err(ctx->err, "cudaEventCreate failed"); return BWTC_CUDA_ECUDA; }
  }
  ctx->timing_detail = detail;
  return 0;
}

int bwtc_cuda_ctx_set_verify(bwtc_cuda_ctx* ctx, int on) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  ctx->verify = on ? 1 : 0;
  return 0;
}

/* Debug / test hooks (declared in include/bwtc_cuda.h): stop after `max_rounds` sort rounds and read
 * back engine buffers so a harness can check every stage against a CPU restatement. */
int bwtc_cuda_ctx_set_debug(bwtc_cuda_ctx* ctx, uint32_t max_rounds) {
  if (!ctx) return BWTC_CUDA_EARG;
  ctx->debug_max_rounds = max_rounds;
  return 0;
}

int bwtc_cuda_debug_read(bwtc_cuda_ctx* ctx, int which, uint64_t offset_bytes, void* dst, uint64_t bytes) {
  if (!ctx || !dst) return BWTC_CUDA_EARG;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return BWTC_CUDA_ECUDA;
  const uint8_t* src = nullptr;
  switch (which) {
    case 0: src = ctx->d_text; break;
    case 1: src = reinterpret_cast<const uint8_t*>(ctx->d_rank); break;
    case 2: src = static_cast<const uint8_t*>(ctx->d_keys[ctx->last_cur]); break;
    case 3: src = reinterpret_cast<const uint8_t*>(ctx->d_idx[ctx->last_cur]); break;
    case 4: src = static_cast<const uint8_t*>(ctx->d_keys[ctx->last_cur ^ 1]); break;
    case 5: src = reinterpret_cast<const uint8_t*>(ctx->d_idx[ctx->last_cur ^ 1]); break;
    case 6: src = reinterpret_cast<const uint8_t*>(ctx->d_zero); break;
    case 7: src = ctx->d_in; break;
#ifdef BWTC_PROFILE_STAGES
    case 8: {
      unsigned long long* pbuf = nullptr;
      CK(ctx, cudaMemcpyFromSymbol(&pbuf, g_prof_buf, sizeof(pbuf)));
      src = reinterpret_cast<const uint8_t*>(pbuf);
      break;
    }
#endif
    default: return BWTC_CUDA_EARG;
  }
  CK(ctx, cudaMemcpy(dst, src + offset_bytes, bytes, cudaMemcpyDeviceToHost));
  return 0;
}

int64_t bwtc_cuda_divbwtf(bwtc_cuda_ctx* ctx, const uint8_t* T, uint8_t* U, uint32_t n, uint32_t* LFpowers,
                          uint32_t nLFpowers, uint32_t* freqs) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!T || !U) { set_err(ctx->err, "null T or U"); return BWTC_CUDA_EARG; }  // divsufsort.c:488
  if (n <= 1) {  // divsufsort.c:489: trivial inputs never reach the sort; LFpowers stays untouched
    if (n == 1) U[0] = T[0];
    return n;
  }
  return run_transform(ctx, false, T, U, nullptr, nullptr, n, LFpowers, nLFpowers, freqs);
}

int64_t bwtc_cuda_divbwt(bwtc_cuda_ctx* ctx, const uint8_t* T, uint8_t* U, uint32_t n, uint32_t* LFpowers,
                         uint32_t nLFpowers) {
  return bwtc_cuda_divbwtf(ctx, T, U, n, LFpowers, nLFpowers, nullptr);
}

int bwtc_cuda_divsufsort(bwtc_cuda_ctx* ctx, const uint8_t* T, int32_t* SA, uint32_t n) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  ctx->err[0] = 0;
  if (!T || !SA) { set_err(ctx->err, "null T or SA"); return BWTC_CUDA_EARG; }  // divsufsort.c: (T == NULL) || (SA == NULL)
  if (n <= 1) {
    if (n == 1) SA[0] = 0;
    return 0;
  }
  if ((uint64_t)n > (uint64_t)ctx->cap + 1) {
    set_err(ctx->err, "raw text of %u bytes exceeds context capacity %u", n, ctx->cap);
    return BWTC_CUDA_ETOOBIG;
  }
  if (!ctx->d_sa) {
    if (cudaSetDevice(ctx->device) != cudaSuccess) { set_err(ctx->err, "cudaSetDevice(%d) failed", ctx->device); return BWTC_CUDA_ECUDA; }
    const size_t bytes = ((size_t)ctx->cap + 1) * 4;
    const cudaError_t e = cudaMalloc((void**)&ctx->d_sa, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      ctx->d_sa = nullptr;
      set_err(ctx->err, "cudaMalloc(%zu bytes) for the suffix array: %s", bytes, cudaGetErrorString(e));
      return BWTC_CUDA_EALLOC;
    }
  }
  return run_divsufsort(ctx, T, nullptr, SA, ctx->d_sa, n);
}

int bwtc_cuda_divsufsort_device(bwtc_cuda_ctx* ctx, const void* d_T, void* d_SA, uint32_t n) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  ctx->err[0] = 0;
  if (!d_T || !d_SA || (reinterpret_cast<uintptr_t>(d_SA) & 3u)) { set_err(ctx->err, "null d_T / d_SA, or d_SA not 4-byte aligned"); return BWTC_CUDA_EARG; }
  if (n == 0) return 0;
  if (n == 1) {
    if (cudaSetDevice(ctx->device) != cudaSuccess) { set_err(ctx->err, "cudaSetDevice(%d) failed", ctx->device); return BWTC_CUDA_ECUDA; }
    CK(ctx, cudaMemsetAsync(d_SA, 0, 4, ctx->stream));
    return host_wait(ctx, ctx->stream) ? BWTC_CUDA_ECUDA : 0;
  }
  return run_divsufsort(ctx, nullptr, static_cast<const uint8_t*>(d_T), nullptr, static_cast<int32_t*>(d_SA), n);
}

int bwtc_cuda_sufcheck(bwtc_cuda_ctx* ctx, const uint8_t* T, const int32_t* SA, uint32_t n) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  ctx->err[0] = 0;
  if (!T || !SA) { set_err(ctx->err, "null T or SA"); return BWTC_CUDA_EARG; }
  if (n == 0) return 0;
  if ((uint64_t)n > (uint64_t)ctx->cap + 1) {
    set_err(ctx->err, "raw text of %u bytes exceeds context capacity %u", n, ctx->cap);
    return BWTC_CUDA_ETOOBIG;
  }
  if (n == 1) {
    if (SA[0] == 0) return 0;
    set_err(ctx->err, "sufcheck: row 0 of 1: value out of range");
    return BWTC_CUDA_ECORRUPT;
  }
  if (cudaSetDevice(ctx->device) != cudaSuccess) { set_err(ctx->err, "cudaSetDevice(%d) failed", ctx->device); return BWTC_CUDA_ECUDA; }
  cudaStream_t st = ctx->stream;
  bwtc_cuda_stats& S = ctx->stats;
  memset(&S, 0, sizeof(S));
  S.n_suffixes = n;
  int32_t* d_SA = static_cast<int32_t*>(ctx->d_keys[1]);  // (8 bytes per suffix; the ISA goes to d_keys[0])
  if (upload(ctx, ctx->d_in, T, n)) return BWTC_CUDA_ECUDA;
  if (upload(ctx, reinterpret_cast<uint8_t*>(d_SA), reinterpret_cast<const uint8_t*>(SA), (size_t)n * 4)) return BWTC_CUDA_ECUDA;
  CK(ctx, cudaEventRecord(ctx->ev_begin, st));
  if (enqueue_sufcheck(ctx, ctx->d_in, d_SA, n)) return BWTC_CUDA_ECUDA;
  CK(ctx, cudaEventRecord(ctx->ev_end, st));
  if (host_wait(ctx, st)) return BWTC_CUDA_ECUDA;
  float ms = 0;
  CK(ctx, cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end));
  S.gpu_ms = ms;
  return sufcheck_failed(ctx, n, "sufcheck") ? BWTC_CUDA_ECORRUPT : 0;
}

int64_t bwtc_cuda_bwt_block(bwtc_cuda_ctx* ctx, uint8_t* block, uint32_t n, uint32_t* LFpowers, uint32_t nLFpowers,
                            uint32_t* freqs) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!block || n == 0) { set_err(ctx->err, "null or empty block"); return BWTC_CUDA_EARG; }
  return run_transform(ctx, true, block, block, nullptr, nullptr, n, LFpowers, nLFpowers, freqs);
}

int64_t bwtc_cuda_bwt_block_runs(bwtc_cuda_ctx* ctx, uint8_t* block, uint32_t n, uint32_t* LFpowers, uint32_t nLFpowers,
                                 uint32_t* freqs, bwtc_cuda_runs* runs) {
  if (runs) runs->count = BWTC_CUDA_RUNS_OVERFLOW;  // (every negative return leaves it so)
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!block || n == 0) { set_err(ctx->err, "null or empty block"); return BWTC_CUDA_EARG; }
  return run_transform(ctx, true, block, block, nullptr, nullptr, n, LFpowers, nLFpowers, freqs, nullptr, runs);
}

int bwtc_cuda_bwt_blocks(bwtc_cuda_ctx* ctx, void* const* blocks, const uint32_t* sizes, uint32_t count, uint32_t starts,
                         int on_device, uint32_t* LFpowers, uint32_t* nLFpowers, uint32_t* freqs) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!blocks || !sizes || !LFpowers || !nLFpowers || count == 0) { set_err(ctx->err, "bad arguments"); return BWTC_CUDA_EARG; }
  for (uint32_t k0 = 0; k0 < count;) {  // runs of at most MAX_BATCH blocks
    uint32_t k1 = std::min<uint32_t>(count, k0 + MAX_BATCH);
    while (k1 > k0 + 1 && !batchable(ctx, sizes + k0, k1 - k0)) --k1;
    const int rc = transform_batch(ctx, const_cast<const void* const*>(blocks + k0), blocks + k0, sizes + k0, k1 - k0, starts,
                                   on_device != 0, LFpowers + (size_t)k0 * 256, nLFpowers + k0,
                                   freqs ? freqs + (size_t)k0 * 256 : nullptr, nullptr);
    if (rc < 0) return rc;
    k0 = k1;
  }
  return 0;
}

int64_t bwtc_cuda_bwt_block_device(bwtc_cuda_ctx* ctx, const void* d_in, void* d_out, uint32_t n, uint32_t* LFpowers,
                                   uint32_t nLFpowers, uint32_t* freqs) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!d_in || !d_out || n == 0) { set_err(ctx->err, "null or empty block"); return BWTC_CUDA_EARG; }
  return run_transform(ctx, true, nullptr, nullptr, static_cast<const uint8_t*>(d_in), static_cast<uint8_t*>(d_out), n,
                       LFpowers, nLFpowers, freqs);
}

int64_t bwtc_cuda_inverse_block(bwtc_cuda_ctx* ctx, uint8_t* block, uint32_t n, const uint32_t* LFpowers, uint32_t nLFpowers) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!block || n == 0 || !LFpowers || nLFpowers < 1) { set_err(ctx->err, "null or empty block / no starting point"); return BWTC_CUDA_EARG; }
  return run_inverse(ctx, true, block, block, nullptr, nullptr, n, LFpowers[0]);
}

int64_t bwtc_cuda_inverse_block_device(bwtc_cuda_ctx* ctx, const void* d_in, void* d_out, uint32_t n, uint32_t eob) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!d_in || !d_out || n == 0) { set_err(ctx->err, "null or empty block"); return BWTC_CUDA_EARG; }
  return run_inverse(ctx, true, nullptr, nullptr, static_cast<const uint8_t*>(d_in), static_cast<uint8_t*>(d_out), n, eob);
}

int bwtc_cuda_inverse_blocks(bwtc_cuda_ctx* ctx, const void* const* in, void* const* out, const uint32_t* sizes, uint32_t count,
                             int on_device, const uint32_t* LFpowers, bwtc_cuda_stats* stats) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!in || !sizes || !LFpowers || count == 0) { set_err(ctx->err, "bad arguments"); return BWTC_CUDA_EARG; }
  std::vector<uint32_t> eobs(count);
  for (uint32_t k = 0; k < count; ++k) eobs[k] = LFpowers[(size_t)k * 256];
  return inverse_blocks(ctx, in, out ? out : const_cast<void* const*>(in), sizes, count, on_device != 0, eobs.data(), stats);
}

int64_t bwtc_cuda_inverse_raw(bwtc_cuda_ctx* ctx, uint8_t* bwt, uint32_t N, const uint32_t* LFpowers, uint32_t nLFpowers) {
  if (!ctx) { set_err(g_err, "null context"); return BWTC_CUDA_EARG; }
  if (!bwt || N < 2 || !LFpowers || nLFpowers < 1) { set_err(ctx->err, "null / too short input or no starting point"); return BWTC_CUDA_EARG; }
  return run_inverse(ctx, false, bwt, bwt, nullptr, nullptr, N, LFpowers[0]);
}

uint32_t bwtc_cuda_num_starting_points(uint32_t block_bytes, uint32_t starts) {
  if (starts < 1) starts = 1; else if (starts > 256) starts = 256;  // BWTManager.cpp:60-64
  return block_bytes <= 256 ? 1u : starts;                         // BWTBlock.cpp:104-108
}

}  // extern "C"

// =====================================================================================================
// Batched look-ahead pipeline: `depth` contexts on one GPU, one persistent host worker per context, a FIFO of
// submitted blocks.  Replaces the synchronous per-slice loop of Compressor::compress (Compressor.cpp:100-109) for the
// BWT stage; results are delivered per block (ticket), so a caller can entropy-code strictly in file order while
// later blocks are still in flight.  Workers sleep on a condition variable when the queue is empty and on blocking-sync
// events while the GPU works: an idle or waiting pipeline costs no host core.
// =====================================================================================================
namespace {
enum PipeKind : int { PIPE_FORWARD = 0, PIPE_INVERSE = 1 };
struct PipeItem {
  int kind = PIPE_FORWARD;
  const void* in = nullptr;
  void* out = nullptr;
  uint32_t n = 0, starts = 0;
  uint32_t eob = 0;         // inverse: the end-of-block row (LFpowers[0] of the forward transform)
  bool on_device = false;
  uint32_t* LF = nullptr;   // 256 words
  uint32_t* nLF = nullptr;
  uint32_t* freqs = nullptr;
  bwtc_cuda_stats* stats = nullptr;
  bwtc_cuda_runs* runs = nullptr;
  uint64_t ticket = 0;
  int rc = 0;
  bool done = false;
};
}  // namespace

struct bwtc_cuda_pipeline {
  int device = 0;
  std::vector<bwtc_cuda_ctx*> ctxs;
  cudaStream_t tstream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<cudaEvent_t> ev_done;
  uint32_t batch_max_block = 0;  // blocks up to this size are batched ...
  uint32_t batch_blocks = 1;     // ... this many at most per batch
  // ---- queue
  std::mutex mu;
  std::condition_variable cv_work, cv_done;
  std::deque<std::shared_ptr<PipeItem>> queue;                       // submitted, not yet claimed (FIFO)
  std::unordered_map<uint64_t, std::shared_ptr<PipeItem>> inflight;  // submitted, not yet waited for
  uint64_t next_ticket = 1;
  bool stopping = false;
  std::vector<std::thread> workers;
  char err[512];
};

namespace {

void pipeline_worker(bwtc_cuda_pipeline* p, bwtc_cuda_ctx* c) {
  cudaSetDevice(p->device);
  std::vector<std::shared_ptr<PipeItem>> grp;
  std::vector<const void*> in;
  std::vector<void*> out;
  std::vector<uint32_t> sizes, nLF, LF, freqs, eobs;
  std::vector<bwtc_cuda_stats> stats;
  for (;;) {
    grp.clear();
    {
      std::unique_lock<std::mutex> lk(p->mu);
      p->cv_work.wait(lk, [&] { return p->stopping || !p->queue.empty(); });
      if (p->queue.empty()) return;  // stopping
      grp.push_back(p->queue.front());
      p->queue.pop_front();
      // consecutive small blocks of equal size (same kind and contract parameters) go to ONE device-side sort / inversion
      if (grp[0]->n <= p->batch_max_block && !grp[0]->runs) {
        sizes.assign(1, grp[0]->n);
        const uint32_t lim = std::min<uint32_t>(MAX_BATCH, p->batch_blocks);
        while (!p->queue.empty() && grp.size() < lim) {
          const PipeItem& nx = *p->queue.front();
          if (nx.kind != grp[0]->kind || nx.on_device != grp[0]->on_device) break;
          if (nx.kind == PIPE_FORWARD &&
              (nx.starts != grp[0]->starts || (nx.freqs == nullptr) != (grp[0]->freqs == nullptr) || nx.runs)) break;
          sizes.push_back(nx.n);
          if (!batchable(c, sizes.data(), (uint32_t)sizes.size())) { sizes.pop_back(); break; }
          grp.push_back(p->queue.front());
          p->queue.pop_front();
        }
      }
    }
    const uint32_t cnt = (uint32_t)grp.size();
    int rc;
    if (grp[0]->kind == PIPE_INVERSE) {
      in.resize(cnt); out.resize(cnt); sizes.resize(cnt); eobs.resize(cnt); stats.resize(cnt);
      for (uint32_t k = 0; k < cnt; ++k) { in[k] = grp[k]->in; out[k] = grp[k]->out; sizes[k] = grp[k]->n; eobs[k] = grp[k]->eob; }
      rc = inverse_blocks(c, in.data(), out.data(), sizes.data(), cnt, grp[0]->on_device, eobs.data(), stats.data());
      if (rc >= 0 || rc == BWTC_CUDA_ECORRUPT)
        for (uint32_t k = 0; k < cnt; ++k)
          if (grp[k]->stats) *grp[k]->stats = stats[k];
    } else if (cnt == 1) {
      PipeItem& it = *grp[0];
      const void* i1 = it.in;
      void* o1 = it.out;
      rc = transform_batch(c, &i1, &o1, &it.n, 1, it.starts, it.on_device, it.LF, it.nLF, it.freqs, it.stats, it.runs);
    } else {
      in.resize(cnt); out.resize(cnt); sizes.resize(cnt); nLF.resize(cnt);
      LF.assign((size_t)cnt * 256, 0u);
      const bool want_freqs = grp[0]->freqs != nullptr;
      if (want_freqs) freqs.assign((size_t)cnt * 256, 0u);
      stats.resize(cnt);
      for (uint32_t k = 0; k < cnt; ++k) { in[k] = grp[k]->in; out[k] = grp[k]->out; sizes[k] = grp[k]->n; }
      rc = transform_batch(c, in.data(), out.data(), sizes.data(), cnt, grp[0]->starts, grp[0]->on_device, LF.data(), nLF.data(),
                           want_freqs ? freqs.data() : nullptr, stats.data());
      if (rc >= 0)
        for (uint32_t k = 0; k < cnt; ++k) {
          PipeItem& it = *grp[k];
          *it.nLF = nLF[k];
          for (uint32_t j = 0; j < nLF[k]; ++j) it.LF[j] = LF[(size_t)k * 256 + j];
          if (want_freqs) for (int ch = 0; ch < 256; ++ch) it.freqs[ch] += freqs[(size_t)k * 256 + ch];
          if (it.stats) *it.stats = stats[k];
        }
    }
    {
      std::lock_guard<std::mutex> lk(p->mu);
      if (rc == BWTC_CUDA_ECORRUPT && grp[0]->kind == PIPE_INVERSE) {
        // only the tickets of the corrupt blocks fail; the rest of the group was restored (DESIGN.md §5.2)
        for (uint32_t k = 0; k < cnt; ++k) {
          PipeItem& it = *grp[k];
          it.rc = (stats[k].flags & 128u) ? BWTC_CUDA_ECORRUPT : 0;
          if (it.rc && !p->err[0])
            set_err(p->err, "block ticket %llu: inverse: not the BWT of any text (with end-of-block row %u)",
                    (unsigned long long)it.ticket, it.eob);
          it.done = true;
        }
      } else {
        if (rc < 0 && !p->err[0]) set_err(p->err, "block ticket %llu (+%u): %s", (unsigned long long)grp[0]->ticket, cnt - 1, c->err);
        for (auto& it : grp) { it->rc = rc < 0 ? rc : 0; it->done = true; }
      }
    }
    p->cv_done.notify_all();
  }
}

uint64_t pipeline_enqueue_locked(bwtc_cuda_pipeline* p, const void* in, void* out, uint32_t n, uint32_t starts, bool on_device,
                                 uint32_t* LF, uint32_t* nLF, uint32_t* freqs, bwtc_cuda_stats* stats, bwtc_cuda_runs* runs = nullptr,
                                 int kind = PIPE_FORWARD, uint32_t eob = 0) {
  auto it = std::make_shared<PipeItem>();
  it->kind = kind; it->eob = eob;
  it->in = in; it->out = out; it->n = n; it->starts = starts; it->on_device = on_device;
  it->LF = LF; it->nLF = nLF; it->freqs = freqs; it->stats = stats; it->runs = runs;
  it->ticket = p->next_ticket++;
  p->queue.push_back(it);
  p->inflight[it->ticket] = it;
  return it->ticket;
}

int pipeline_wait_ticket(bwtc_cuda_pipeline* p, uint64_t ticket) {
  std::unique_lock<std::mutex> lk(p->mu);
  auto f = p->inflight.find(ticket);
  if (f == p->inflight.end()) { set_err(p->err, "unknown ticket %llu", (unsigned long long)ticket); return BWTC_CUDA_EARG; }
  std::shared_ptr<PipeItem> it = f->second;
  p->cv_done.wait(lk, [&] { return it->done; });
  p->inflight.erase(ticket);
  return it->rc;
}

}  // namespace

extern "C" {

void bwtc_cuda_pipeline_destroy(bwtc_cuda_pipeline* p) {
  if (!p) return;
  {
    std::lock_guard<std::mutex> lk(p->mu);
    p->stopping = true;
    p->queue.clear();
  }
  p->cv_work.notify_all();
  for (std::thread& t : p->workers) t.join();
  cudaSetDevice(p->device);
  for (bwtc_cuda_ctx* c : p->ctxs) ctx_free(c);
  for (cudaEvent_t e : p->ev_done) cudaEventDestroy(e);
  if (p->ev0) cudaEventDestroy(p->ev0);
  if (p->ev1) cudaEventDestroy(p->ev1);
  if (p->tstream) cudaStreamDestroy(p->tstream);
  delete p;
}

int bwtc_cuda_pipeline_create(bwtc_cuda_pipeline** out, int device, int depth, uint32_t max_block_bytes) {
  if (!out || depth < 1 || depth > 64) { set_err(g_err, "bad arguments"); return BWTC_CUDA_EARG; }
  *out = nullptr;
  bwtc_cuda_pipeline* p = new (std::nothrow) bwtc_cuda_pipeline();
  if (!p) return BWTC_CUDA_EALLOC;
  p->device = device;
  p->err[0] = 0;
  // Small blocks: give every context room for a batch of them (~32 MiB of text, at most MAX_BATCH blocks), so a
  // worker sorts e.g. 32 x 1 MiB blocks as one problem instead of 32 launch-latency-bound ones.
  uint64_t cap = max_block_bytes;
  {
    uint64_t target = 32ull << 20;
    if (const char* e = getenv("BWTC_BATCH_MIB")) { const long v = atol(e); target = v > 0 ? (uint64_t)v << 20 : 0; }
    const char* eb = getenv("BWTC_BATCH");
    if ((!eb || atoi(eb) != 0) && max_block_bytes > 0 && (uint64_t)max_block_bytes * 4 <= target) {  // blocks <= 8 MiB
      uint64_t nb = target / max_block_bytes;
      if (nb > MAX_BATCH) nb = MAX_BATCH;
      p->batch_blocks = (uint32_t)nb;
      p->batch_max_block = max_block_bytes;
      cap = (uint64_t)max_block_bytes * nb + nb;
    }
  }
  for (int i = 0; i < depth; ++i) {
    bwtc_cuda_ctx* c = nullptr;
    int rc = bwtc_cuda_ctx_create(&c, device, (uint32_t)cap);
    if (rc) { bwtc_cuda_pipeline_destroy(p); return rc; }
    p->ctxs.push_back(c);
  }
  bool ok = cudaStreamCreateWithFlags(&p->tstream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreate(&p->ev0) == cudaSuccess && cudaEventCreateWithFlags(&p->ev1, cudaEventBlockingSync) == cudaSuccess;
  p->ev_done.resize(depth, nullptr);
  for (int i = 0; ok && i < depth; ++i) ok = cudaEventCreateWithFlags(&p->ev_done[i], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) { set_err(g_err, "pipeline stream/event creation failed"); bwtc_cuda_pipeline_destroy(p); return BWTC_CUDA_ECUDA; }
  for (bwtc_cuda_ctx* c : p->ctxs) p->workers.emplace_back(pipeline_worker, p, c);
  *out = p;
  return 0;
}

const char* bwtc_cuda_pipeline_error(const bwtc_cuda_pipeline* p) { return p ? p->err : g_err; }

int bwtc_cuda_pipeline_set_round0(bwtc_cuda_pipeline* p, uint32_t chars, uint32_t key_bytes) {
  if (!p) return BWTC_CUDA_EARG;
  for (bwtc_cuda_ctx* c : p->ctxs) {
    int rc = bwtc_cuda_ctx_set_round0(c, chars, key_bytes);
    if (rc) return rc;
  }
  return 0;
}

int bwtc_cuda_pipeline_set_timing(bwtc_cuda_pipeline* p, int detail) {
  if (!p) return BWTC_CUDA_EARG;
  for (bwtc_cuda_ctx* c : p->ctxs) {
    int rc = bwtc_cuda_ctx_set_timing(c, detail);
    if (rc) return rc;
  }
  return 0;
}

int bwtc_cuda_pipeline_set_verify(bwtc_cuda_pipeline* p, int on) {
  if (!p) { set_err(g_err, "null pipeline"); return BWTC_CUDA_EARG; }
  for (bwtc_cuda_ctx* c : p->ctxs) c->verify = on ? 1 : 0;
  return 0;
}

int bwtc_cuda_pipeline_submit(bwtc_cuda_pipeline* p, const uint8_t* in, uint8_t* out, uint32_t n, uint32_t starts,
                              int on_device, uint32_t* LFpowers, uint32_t* nLF, uint32_t* freqs, bwtc_cuda_stats* stats,
                              uint64_t* ticket) {
  if (!p || !in || !out || !LFpowers || !nLF || !ticket || n == 0) { if (p) set_err(p->err, "bad arguments"); return BWTC_CUDA_EARG; }
  {
    std::lock_guard<std::mutex> lk(p->mu);
    *ticket = pipeline_enqueue_locked(p, in, out, n, starts, on_device != 0, LFpowers, nLF, freqs, stats);
  }
  p->cv_work.notify_one();
  return 0;
}

int bwtc_cuda_pipeline_submit_runs(bwtc_cuda_pipeline* p, const uint8_t* in, uint8_t* out, uint32_t n, uint32_t starts,
                                   uint32_t* LFpowers, uint32_t* nLF, uint32_t* freqs, bwtc_cuda_runs* runs, uint64_t* ticket) {
  if (runs) runs->count = BWTC_CUDA_RUNS_OVERFLOW;  // (stays so unless the block succeeds)
  if (!p || !in || !out || !LFpowers || !nLF || !ticket || n == 0) { if (p) set_err(p->err, "bad arguments"); return BWTC_CUDA_EARG; }
  {
    std::lock_guard<std::mutex> lk(p->mu);
    *ticket = pipeline_enqueue_locked(p, in, out, n, starts, false, LFpowers, nLF, freqs, nullptr, runs);
  }
  p->cv_work.notify_one();
  return 0;
}

int bwtc_cuda_pipeline_submit_inverse(bwtc_cuda_pipeline* p, const uint8_t* in, uint8_t* out, uint32_t n, uint32_t eob,
                                      int on_device, bwtc_cuda_stats* stats, uint64_t* ticket) {
  if (!p) { set_err(g_err, "null pipeline"); return BWTC_CUDA_EARG; }
  if (!in || !out || !ticket || n == 0) { set_err(p->err, "bad arguments"); return BWTC_CUDA_EARG; }
  if (eob > n) { set_err(p->err, "inverse: end-of-block position %u outside [0, %u)", eob, n + 1u); return BWTC_CUDA_EARG; }
  {
    std::lock_guard<std::mutex> lk(p->mu);
    *ticket = pipeline_enqueue_locked(p, in, out, n, 0, on_device != 0, nullptr, nullptr, nullptr, stats, nullptr, PIPE_INVERSE, eob);
  }
  p->cv_work.notify_one();
  return 0;
}

int bwtc_cuda_pipeline_wait(bwtc_cuda_pipeline* p, uint64_t ticket) {
  if (!p) return BWTC_CUDA_EARG;
  return pipeline_wait_ticket(p, ticket);
}

int bwtc_cuda_pipeline_run(bwtc_cuda_pipeline* p, const uint8_t* const* in, uint8_t* const* out, const uint32_t* sizes,
                           uint32_t nblocks, uint32_t starts, int on_device, uint32_t* LFpowers, uint32_t* nLF,
                           uint32_t* freqs, bwtc_cuda_stats* stats) {
  if (!p || !in || !out || !sizes || !LFpowers || !nLF) { if (p) set_err(p->err, "bad arguments"); return BWTC_CUDA_EARG; }
  for (uint32_t i = 0; i < nblocks; ++i)
    if (!in[i] || !out[i] || sizes[i] == 0) { set_err(p->err, "null or empty block %u", i); return BWTC_CUDA_EARG; }
  std::vector<uint64_t> tickets(nblocks);
  {
    // all blocks are queued before any worker wakes up, so runs of small blocks are grouped deterministically
    std::lock_guard<std::mutex> lk(p->mu);
    p->err[0] = 0;
    for (uint32_t i = 0; i < nblocks; ++i)
      tickets[i] = pipeline_enqueue_locked(p, in[i], out[i], sizes[i], starts, on_device != 0, LFpowers + (size_t)i * 256, nLF + i,
                                           freqs ? freqs + (size_t)i * 256 : nullptr, stats ? stats + i : nullptr);
  }
  p->cv_work.notify_all();
  int first_err = 0;
  for (uint32_t i = 0; i < nblocks; ++i) {
    const int rc = pipeline_wait_ticket(p, tickets[i]);
    if (rc < 0 && !first_err) first_err = rc;
  }
  return first_err;
}

int bwtc_cuda_pipeline_timing_begin(bwtc_cuda_pipeline* p) {
  if (!p) return BWTC_CUDA_EARG;
  if (cudaSetDevice(p->device) != cudaSuccess) return BWTC_CUDA_ECUDA;
  if (cudaEventRecord(p->ev0, p->tstream) != cudaSuccess) return BWTC_CUDA_ECUDA;
  for (bwtc_cuda_ctx* c : p->ctxs)
    if (cudaStreamWaitEvent(c->stream, p->ev0, 0) != cudaSuccess) return BWTC_CUDA_ECUDA;
  return 0;
}

float bwtc_cuda_pipeline_timing_end(bwtc_cuda_pipeline* p) {
  if (!p) return (float)BWTC_CUDA_EARG;
  if (cudaSetDevice(p->device) != cudaSuccess) return (float)BWTC_CUDA_ECUDA;
  for (size_t i = 0; i < p->ctxs.size(); ++i) {
    if (cudaEventRecord(p->ev_done[i], p->ctxs[i]->stream) != cudaSuccess) return (float)BWTC_CUDA_ECUDA;
    if (cudaStreamWaitEvent(p->tstream, p->ev_done[i], 0) != cudaSuccess) return (float)BWTC_CUDA_ECUDA;
  }
  if (cudaEventRecord(p->ev1, p->tstream) != cudaSuccess) return (float)BWTC_CUDA_ECUDA;
  if (cudaEventSynchronize(p->ev1) != cudaSuccess) return (float)BWTC_CUDA_ECUDA;
  float ms = 0;
  if (cudaEventElapsedTime(&ms, p->ev0, p->ev1) != cudaSuccess) return (float)BWTC_CUDA_ECUDA;
  return ms;
}

}  // extern "C"
