/* include/bwtc_cuda.h — C-ABI of the B200-native forward Burrows-Wheeler transform engine for bwtc.
 *
 * This is the drop-in boundary for ONE hot path of pjmikkol/bwtc: the per-block forward BWT that the
 * reference computes with its modified divsufsort / SA-IS behind bwtransforms/BWTransform.  Plain
 * pointers and sizes only; no C++/torch types.  Implemented by bwtc_b200/libbwtc_cuda.so
 * (bwtc_b200/csrc/bwt_engine.cu, hand-written sm_100a kernels).  There is no CPU fallback: every entry
 * point fails loudly (negative return + bwtc_cuda_last_error) if the device or a kernel fails.
 *
 * Reference interfaces replaced (paths relative to the reference tree):
 *   bwtc_cuda_divbwt / bwtc_cuda_divbwtf   <-  divbwt / divbwtf          bwtransforms/divsufsort.h:86-94,
 *                                              bwtransforms/divsufsort.c:440-522 (as called by
 *                                              Divsufsorter::doTransform, bwtransforms/Divsufsorter.hpp:54-65)
 *   bwtc_cuda_divsufsort / _device /       <-  divsufsort / sufcheck                  bwtransforms/divsufsort.h (the
 *   bwtc_cuda_sufcheck                         library's suffix-array entry point and its checker, beside the BWT
 *                                              entry points above)
 *   bwtc_cuda_bwt_block                    <-  BWTransform::doTransform(BWTBlock&, uint32 freqs[256])
 *                                              bwtransforms/BWTransform.cpp:39-64 (reverse / sentinel /
 *                                              hole-fill fused on the device)
 *   bwtc_cuda_num_starting_points          <-  BWTManager::setStartingPoints + BWTBlock::prepareLFpowers
 *                                              bwtransforms/BWTManager.cpp:60-64, BWTBlock.cpp:104-108
 *   bwtc_cuda_inverse_block / _raw         <-  InverseBWTransform::doTransform(BWTBlock&) / (byte*, uint32, LFpow)
 *                                              bwtransforms/InverseBWT.cpp:47-51, InverseBWT.hpp:49-50 (MtlSaInverseBWT.cpp)
 *   bwtc_cuda_inverse_blocks /             <-  the per-slice InverseBWTransform::doTransform calls of
 *   bwtc_cuda_pipeline_submit_inverse          Decompressor::decompress (Decompressor.cpp:58-94, InverseBWT.cpp:47-51):
 *                                              equal-sized slices inverted as one device-side problem, or streamed
 *   bwtc_cuda_pipeline_*                   <-  the per-slice loop of Compressor::compress
 *                                              Compressor.cpp:100-109 (independent BWT blocks), batched
 *                                              with look-ahead over several in-flight blocks per GPU
 */
#ifndef BWTC_CUDA_H_
#define BWTC_CUDA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Return codes (all entry points that return int / int64_t): >= 0 success. */
#define BWTC_CUDA_EARG      (-1)  /* bad arguments (same meaning as divbwtf's -1, divsufsort.c:488) */
#define BWTC_CUDA_EALLOC    (-2)  /* host or device allocation failed (divbwtf's -2, divsufsort.c:513-515) */
#define BWTC_CUDA_ECUDA     (-3)  /* a CUDA runtime call or kernel failed */
#define BWTC_CUDA_EINTERNAL (-4)  /* internal consistency check failed (e.g. look-back watchdog) */
#define BWTC_CUDA_ETOOBIG   (-5)  /* block larger than the context capacity / engine limit */
#define BWTC_CUDA_ECORRUPT  (-6)  /* inverse: the input is not the BWT of any text (with this end-of-block row); the message
                                   * names the block */
#define BWTC_CUDA_EVERIFY   (-7)  /* forward with verification on: the output did not restore the input (see
                                   * bwtc_cuda_ctx_set_verify); every caller buffer still holds its input */

/* Largest block (bytes, excluding the sentinel slot) the engine accepts: the reference's own limit — blocks below
 * 2^31 - 2 bytes (Compressor.cpp:78-79, PrecompressorBlock.cpp:126; N = n + 1 suffixes must index with 31 bits because
 * LFpowers are serialised as 31-bit values, BWTBlock.cpp:61-86). */
#define BWTC_CUDA_MAX_BLOCK ((uint32_t)0x7FFFFFFDu)

/* Device scratch per suffix (input, text, output, rank, two key + two id buffers, staged ranks, payload bytes, status
 * words) — an upper bound for blocks of 1 MiB and more; bwtc_cuda_scratch_bytes(n) is the exact figure a context for n-byte blocks allocates. */
#define BWTC_CUDA_SCRATCH_BYTES_PER_SUFFIX 40
#define BWTC_CUDA_SCRATCH_FIXED_BYTES (8u << 20)  /* + tables that do not grow with the block (status pad rows, sample and prefix tables) */

typedef struct bwtc_cuda_ctx bwtc_cuda_ctx;           /* one stream + device scratch for one in-flight block */
typedef struct bwtc_cuda_pipeline bwtc_cuda_pipeline; /* several contexts + host workers on one GPU */

/* Per-block execution record, filled by every transform (so a harness can recompute the algorithmic
 * bytes of SURVEY.md §8d / DESIGN.md: rounds, live suffix counts m_r, digit passes P_r). */
#define BWTC_CUDA_MAX_ROUNDS 40
typedef struct bwtc_cuda_stats {
  uint32_t n_suffixes;                      /* N = block bytes + 1 (block contract) or n (raw contract) */
  uint32_t sigma;                           /* distinct byte values */
  uint32_t bits_per_char;                   /* dense code width b */
  uint32_t chars_round0;                    /* c: characters packed into the round-0 key */
  uint32_t key_bytes_round0;                /* 4 or 8 */
  uint32_t rounds;                          /* sort rounds executed, round 0 included */
  uint32_t live[BWTC_CUDA_MAX_ROUNDS];      /* m_r: records sorted in round r (m_0 = N) */
  uint32_t passes[BWTC_CUDA_MAX_ROUNDS];    /* P_r: radix digit passes executed in round r */
  uint32_t prefix_len[BWTC_CUDA_MAX_ROUNDS];/* h_r: prefix length already ordered when round r starts */
  uint64_t kernel_launches;                 /* kernels launched for this block */
  uint64_t algorithmic_bytes;               /* B_alg of this block per DESIGN.md §4 */
  float    gpu_ms;                          /* device time first kernel -> last kernel (CUDA events) */
  float    sort_ms;                         /* device time inside radix digit passes (only with detailed timing on) */
  uint64_t sort_bytes;                      /* algorithmic bytes moved by the radix digit passes */
  uint32_t sort_launches;                   /* radix digit pass launches */
  uint32_t sort0_launches;                  /* ... of which round-0 passes (all N records each) */
  uint64_t sort0_bytes;                     /* algorithmic bytes moved by the round-0 passes */
  float    sort0_ms;                        /* device time inside the round-0 passes (detailed timing on) */
  uint32_t flags;            /* bit 0: look-back kernels ran with ticket counters (watchdog fallback or BWTC_STATIC_TILES=0);
                              * bit 1: the blocks of a batch were sorted as one text; bit 2: predecessor codes packed above the ids;
                              * bit 3: ... carried as a one-byte payload array; bit 6: the forward output (block or raw
                              * contract) and its LFpowers were verified by a device-side inversion (bwtc_cuda_ctx_set_verify,
                              * BWTC_VERIFY; for bwtc_cuda_divsufsort: its suffix array passed the device-side sufcheck); bit 7:
                              * inverse only, this block is corrupt (BWTC_CUDA_ECORRUPT); bit 8: this call produced a suffix
                              * array (bwtc_cuda_divsufsort, _device) */
  uint32_t batch_blocks;     /* blocks this record describes: 1, or the size of the batch that was sorted as one text (every
                              * block of the batch then carries the SAME record — count it once; flags bit 7 is the one field
                              * in which the records of one inverse batch may differ) */
} bwtc_cuda_stats;

/* ---- library / device ------------------------------------------------------------------------ */
int         bwtc_cuda_device_count(void);           /* number of CUDA devices, or BWTC_CUDA_ECUDA */
const char* bwtc_cuda_version(void);
uint32_t    bwtc_cuda_stats_sizeof(void);           /* sizeof(bwtc_cuda_stats) the library was built with */
/* Thread-local message of the last failing call that had no context to attach it to. */
const char* bwtc_cuda_global_error(void);

/* ---- context ------------------------------------------------------------------------------------ */
/* Allocates streams, device scratch (BWTC_CUDA_SCRATCH_BYTES_PER_SUFFIX bytes per suffix) and small pinned buffers for
 * blocks up to max_block_bytes on `device` (raw texts up to max_block_bytes + 1: the same max_block_bytes + 1 suffixes).
 * Replaces the per-call malloc of divbwtf (divsufsort.c:491-493). */
int         bwtc_cuda_ctx_create(bwtc_cuda_ctx** out, int device, uint32_t max_block_bytes);
uint64_t    bwtc_cuda_scratch_bytes(uint32_t max_block_bytes);  /* device bytes such a context allocates */
void        bwtc_cuda_ctx_destroy(bwtc_cuda_ctx* ctx);
const char* bwtc_cuda_last_error(const bwtc_cuda_ctx* ctx);
int         bwtc_cuda_get_stats(const bwtc_cuda_ctx* ctx, bwtc_cuda_stats* out);
/* Tuning knobs (0 = automatic): force the number of characters / key bytes of the round-0 key. */
int         bwtc_cuda_ctx_set_round0(bwtc_cuda_ctx* ctx, uint32_t chars, uint32_t key_bytes);
/* detail != 0: bracket every radix digit pass with CUDA events on the context's stream so that
 * stats.sort_ms / sort_bytes / sort_launches give the dominant kernel's average launch duration. */
int         bwtc_cuda_ctx_set_timing(bwtc_cuda_ctx* ctx, int detail);
/* on != 0: every forward call (bwtc_cuda_bwt_block, _device, _runs, bwtc_cuda_bwt_blocks, and the raw bwtc_cuda_divbwt /
 * divbwtf) is verified before it returns: the device inverts its device-resident output (end-of-block rows from the
 * device-side LFpowers, a batch as one batched inversion, a raw text with its own last byte as the key of its end-of-text
 * row) and compares the result with the input, which the device still holds; every LFpowers entry (LFpowers[j],
 * 1 <= j < nLFpowers, of every block) is checked against the row the inversion visits at its text position.  On a mismatch
 * the call returns BWTC_CUDA_EVERIFY and every caller buffer holds its input: host outputs (a raw U, aliasing T or not),
 * LFpowers and freqs are written only after the host has read the check word, and an in-place device block is rewritten
 * from the device copy (a device output that does not alias its input, and the run arrays of bwtc_cuda_bwt_block_runs,
 * are then unspecified).  Costs about one inverse transform and one host wait per call; stats.flags bit 6 marks a verified
 * block, stats.gpu_ms includes the check.  Raw texts of n <= 1 bytes return early, unverified.  Off (0) by default; the
 * environment variable BWTC_VERIFY=1, read when a context is created, makes on the initial value of every context (and
 * so of every pipeline and host-side class), which this call still overrides per context.  Off, every call runs exactly
 * the kernels it runs without this switch.  The context stays usable after BWTC_CUDA_EVERIFY. */
int         bwtc_cuda_ctx_set_verify(bwtc_cuda_ctx* ctx, int on);
/* Debug / test hooks: max_rounds != 0 stops the refinement after that many sort rounds (the output is
 * then deliberately incomplete); bwtc_cuda_debug_read copies an engine buffer to the host
 * (which: 0 text, 1 rank[], 2/3 sorted keys/ids of the last round, 4/5 the other sort buffer,
 * 6 control+histogram words, 7 staged input). */
int         bwtc_cuda_ctx_set_debug(bwtc_cuda_ctx* ctx, uint32_t max_rounds);
int         bwtc_cuda_debug_read(bwtc_cuda_ctx* ctx, int which, uint64_t offset_bytes, void* dst, uint64_t bytes);

/* ---- raw contract: same seven logical arguments as divbwtf (divsufsort.h:91-94) ------------------ */
/* T: n input bytes (host).  U: n output bytes (host, may alias T).  Computes the BWT of T under the
 * "implicit end sentinel, shorter suffix first" order divsufsort realises: pidx = rank of suffix 0,
 * U[r] = T[SA[r]-1] for r != pidx, U[pidx] is left untouched, LFpowers[0] = pidx,
 * LFpowers[j] = rank of suffix n - j*(n / nLFpowers), and freqs[U[r]] is INCREMENTED for r != pidx
 * (freqs may be NULL = divbwt).  n <= 1: U[0] = T[0], LFpowers untouched, returns n (divsufsort.c:489).
 * Returns pidx. */
int64_t bwtc_cuda_divbwtf(bwtc_cuda_ctx* ctx, const uint8_t* T, uint8_t* U, uint32_t n,
                          uint32_t* LFpowers, uint32_t nLFpowers, uint32_t* freqs);
int64_t bwtc_cuda_divbwt(bwtc_cuda_ctx* ctx, const uint8_t* T, uint8_t* U, uint32_t n,
                         uint32_t* LFpowers, uint32_t nLFpowers);

/* ---- suffix array of a raw text: libdivsufsort's divsufsort / sufcheck (divsufsort.h) ------------- */
/* divsufsort(T, SA, n): SA[0..n) = the suffix array of T under the raw contract's order (implicit end sentinel, a suffix
 * that is a prefix of another sorts first) -- the order bwtc_cuda_divbwtf's output is defined by (U[r] = T[SA[r]-1],
 * pidx = the row of suffix 0).  Returns 0 or a negative error (-1 / -2 keep divsufsort's meaning).  n == 0: nothing;
 * n == 1: SA[0] = 0 (the host variant does not touch the device).  n <= max_block_bytes + 1 (else BWTC_CUDA_ETOOBIG).
 * T and SA may be pageable or pinned host memory: pinned SA is copied directly, pageable SA through the context's pinned
 * staging ring.  The SA is written on the device where each suffix becomes unique, beside its BWT byte.  Memory: the host
 * variant allocates a 4 (max_block_bytes + 1)-byte device array on its first call (BWTC_CUDA_EALLOC if that fails, the
 * context stays usable), freed by bwtc_cuda_ctx_destroy -- on top of bwtc_cuda_scratch_bytes; _device emits straight into
 * d_SA (n int32 entries, 4-byte aligned, else BWTC_CUDA_EARG) and allocates nothing.  With verification on
 * (bwtc_cuda_ctx_set_verify, BWTC_VERIFY) the device runs the sufcheck below on the SA before anything reaches the caller:
 * on a failure the call returns BWTC_CUDA_EVERIFY, a host SA is untouched, a d_SA holds unspecified values.
 * stats.flags bit 8 is set (bit 6 too when verified); no other entry point sets bit 8. */
int bwtc_cuda_divsufsort(bwtc_cuda_ctx* ctx, const uint8_t* T, int32_t* SA, uint32_t n);
int bwtc_cuda_divsufsort_device(bwtc_cuda_ctx* ctx, const void* d_T, void* d_SA, uint32_t n);  /* d_SA 4-byte aligned */
/* sufcheck(T, SA, n): 0 if SA (host, pageable or pinned) is the suffix array of T, BWTC_CUDA_ECORRUPT if not -- the message
 * names the first offending row and why: out of range / duplicate (of an earlier row) / out of order; range and duplicate
 * failures are reported before order failures.  Other negatives as usual (BWTC_CUDA_ETOOBIG above max_block_bytes + 1).
 * Unlike libdivsufsort's sequential sufcheck, which returns -2 / -3 / -4 for the three kinds of failure, one code is used:
 * those values are BWTC_CUDA_EALLOC / ECUDA / EINTERNAL here.  Runs in the context's scratch (stats: gpu_ms = the check). */
int bwtc_cuda_sufcheck(bwtc_cuda_ctx* ctx, const uint8_t* T, const int32_t* SA, uint32_t n);

/* ---- block contract: BWTransform::doTransform(BWTBlock&, freqs) (BWTransform.cpp:52-64) ---------- */
/* block: n bytes (host), transformed IN PLACE; unlike the reference wrapper the byte after the block
 * is never touched.  LFpowers must hold nLFpowers = bwtc_cuda_num_starting_points(n, starts) entries.
 * freqs (256 counters, incremented) may be NULL.  Returns pidx = LFpowers[0]. */
int64_t bwtc_cuda_bwt_block(bwtc_cuda_ctx* ctx, uint8_t* block, uint32_t n,
                            uint32_t* LFpowers, uint32_t nLFpowers, uint32_t* freqs);
/* Same transform with input and output already resident in device memory (d_in, d_out: n bytes each,
 * may alias).  LFpowers / freqs are host pointers.  Used to measure kernel-only throughput. */
int64_t bwtc_cuda_bwt_block_device(bwtc_cuda_ctx* ctx, const void* d_in, void* d_out, uint32_t n,
                                   uint32_t* LFpowers, uint32_t nLFpowers, uint32_t* freqs);
/* Several blocks of one precompressor block (the slices Compressor::compress walks, Compressor.cpp:100-109)
 * through one context, each transformed IN PLACE exactly as bwtc_cuda_bwt_block would.  blocks[k]: sizes[k] bytes, host
 * pointers (on_device = 0) or device pointers (on_device != 0).  LFpowers: count x 256 words, row k receives
 * nLFpowers[k] = bwtc_cuda_num_starting_points(sizes[k], starts) entries; freqs: count x 256 counters (incremented)
 * or NULL.  Runs of 2..BWTC_CUDA_MAX_BATCH blocks of EQUAL size (the last of a run may be shorter) that fit the
 * context's capacity together (sum of sizes + count <= max_block_bytes + 1) are sorted as ONE device-side problem —
 * small blocks stop being launch-latency-bound (SURVEY.md §8e "small blocks are batched per launch"); other
 * blocks are processed one after the other.  The results do not depend on the grouping.  Returns 0 or an error. */
#define BWTC_CUDA_MAX_BATCH 64
int bwtc_cuda_bwt_blocks(bwtc_cuda_ctx* ctx, void* const* blocks, const uint32_t* sizes, uint32_t count,
                         uint32_t starts, int on_device, uint32_t* LFpowers, uint32_t* nLFpowers, uint32_t* freqs);
/* ---- run statistics of the transformed block (SURVEY.md §8f, row f3) -------------------------------------------- */
/* The maximal runs of equal bytes of the n output bytes, in order: symbol[k], start[k] (start[0] = 0; run k ends where
 * run k+1 starts, the last one at n).  This is what HuffmanEncoder::encodeData obtains per section by re-scanning the
 * block (utils::calculateRunFrequenciesAndStoreRuns, Utils.cpp:150-170; "TODO: Also gather information about the runs
 * during BWT", HuffmanCoders.cpp:54); the host slices the runs at its section boundaries.  The caller provides the two
 * arrays and their capacity; if the block has more runs than that, count = BWTC_CUDA_RUNS_OVERFLOW and the arrays are
 * left alone (text-like blocks have ~0.75 runs per byte: scanning on the host is then cheaper than 5 bytes per run over
 * PCIe — pass a capacity of n/8 or so and fall back to the scan on overflow).  A NULL symbol or start array counts as
 * overflow.  Every negative return (arguments, capacity, BWTC_CUDA_EVERIFY, ...) also leaves count =
 * BWTC_CUDA_RUNS_OVERFLOW, so a caller that only looks at count never takes the runs of a failed block; the arrays are
 * then untouched, except after BWTC_CUDA_EVERIFY, which leaves them unspecified.  On success the entries from index count
 * on are untouched. */
#define BWTC_CUDA_RUNS_OVERFLOW 0xFFFFFFFFu
typedef struct bwtc_cuda_runs {
  uint32_t  capacity;  /* in : runs the arrays can hold */
  uint32_t  count;     /* out: number of runs, or BWTC_CUDA_RUNS_OVERFLOW */
  uint8_t*  symbol;    /* out: capacity bytes (host) */
  uint32_t* start;     /* out: capacity words (host) */
} bwtc_cuda_runs;
/* bwtc_cuda_bwt_block + the runs of its output. */
int64_t bwtc_cuda_bwt_block_runs(bwtc_cuda_ctx* ctx, uint8_t* block, uint32_t n, uint32_t* LFpowers, uint32_t nLFpowers,
                                 uint32_t* freqs, bwtc_cuda_runs* runs);

/* ---- inverse transform (SURVEY.md §8f, row f4): InverseBWTransform::doTransform (InverseBWT.hpp:45-55) ---------------- */
/* Block level (InverseBWT.cpp:47-51): block holds the n bytes a forward block transform produced, LFpowers its starting
 * points (only LFpowers[0], the end-of-block position, is needed: the device makes its own, far denser samples).  The
 * original n bytes are restored IN PLACE; the byte after the block is never touched.  Returns n.
 * Every inverse entry point checks that its input is the BWT of some text with that end-of-block row (exactly: the
 * permutation it defines is one cycle) and returns BWTC_CUDA_ECORRUPT if not.  A pageable host block is then untouched; a
 * pinned host or device output (written speculatively, so that a valid block costs no extra wait) holds unspecified bytes. */
int64_t bwtc_cuda_inverse_block(bwtc_cuda_ctx* ctx, uint8_t* block, uint32_t n, const uint32_t* LFpowers, uint32_t nLFpowers);
int64_t bwtc_cuda_inverse_block_device(bwtc_cuda_ctx* ctx, const void* d_in, void* d_out, uint32_t n, uint32_t eob);
/* Raw virtual doTransform(byte* bwt, uint32 N, LFpow) (InverseBWT.hpp:49-50): bwt[0..N) = L with bwt[LFpowers[0]] ignored;
 * on return bwt[0..N-1) is the original block (bwt[N-1] is left as it was).  Returns N-1. */
int64_t bwtc_cuda_inverse_raw(bwtc_cuda_ctx* ctx, uint8_t* bwt, uint32_t N, const uint32_t* LFpowers, uint32_t nLFpowers);
/* Several blocks through one context, each restored exactly as bwtc_cuda_inverse_block would: in[k] holds the sizes[k]
 * bytes a forward block transform produced, the original bytes land in out[k] (out may be NULL: in place; out[k] may alias
 * in[k]).  Host pointers, or device pointers when on_device != 0.  LFpowers: count x 256 words in the layout
 * bwtc_cuda_bwt_blocks / bwtc_cuda_pipeline_run produce; only LFpowers[k*256] (block k's end-of-block row) is read.  Runs
 * that qualify as for bwtc_cuda_bwt_blocks (2..BWTC_CUDA_MAX_BATCH blocks of equal size, the last may be shorter, together
 * within the context's capacity) are inverted as ONE device-side problem — whatever byte values the blocks contain —
 * others one after the other.  The byte after each block is never touched.  Every argument is checked before any work.
 * stats: count records (the blocks of a batch share one, batch_blocks = its size, flags bit 1 set) or NULL.
 * Corrupt blocks do not stop the call: every valid block is restored, the buffer of each corrupt block is left untouched
 * (whatever its kind), its record gets flags bit 7, and the call returns BWTC_CUDA_ECORRUPT naming the first one.
 * Returns 0 or a negative error. */
int bwtc_cuda_inverse_blocks(bwtc_cuda_ctx* ctx, const void* const* in, void* const* out, const uint32_t* sizes,
                             uint32_t count, int on_device, const uint32_t* LFpowers, bwtc_cuda_stats* stats);
/* BWTManager::setStartingPoints clamp + BWTBlock::prepareLFpowers sizing. */
uint32_t bwtc_cuda_num_starting_points(uint32_t block_bytes, uint32_t starts);

/* ---- batched pipeline over independent blocks (one GPU) ------------------------------------------- */
/* `depth` contexts (in-flight blocks) on `device`, each with a host worker thread; blocks are handed
 * out in order and may complete out of order, results land in the caller's arrays by block index. */
int  bwtc_cuda_pipeline_create(bwtc_cuda_pipeline** out, int device, int depth, uint32_t max_block_bytes);
void bwtc_cuda_pipeline_destroy(bwtc_cuda_pipeline* p);
const char* bwtc_cuda_pipeline_error(const bwtc_cuda_pipeline* p);
int  bwtc_cuda_pipeline_set_round0(bwtc_cuda_pipeline* p, uint32_t chars, uint32_t key_bytes);
int  bwtc_cuda_pipeline_set_timing(bwtc_cuda_pipeline* p, int detail);
/* bwtc_cuda_ctx_set_verify on every context of the pipeline: forward blocks (run, submit, submit_runs) are verified.
 * Its contexts start from BWTC_VERIFY like any other. */
int  bwtc_cuda_pipeline_set_verify(bwtc_cuda_pipeline* p, int on);
/* Transforms nblocks blocks.  in[i]/out[i]: sizes[i] bytes each (may alias; host memory, or device
 * memory when on_device != 0).  LFpowers: nblocks x 256 uint32 (row i gets nLF[i] entries, where
 * nLF[i] = bwtc_cuda_num_starting_points(sizes[i], starts) is written by the call); freqs: nblocks x 256
 * uint32 incremented per block, or NULL; stats: nblocks records or NULL.
 * Returns 0, or the first negative error. */
int  bwtc_cuda_pipeline_run(bwtc_cuda_pipeline* p, const uint8_t* const* in, uint8_t* const* out,
                            const uint32_t* sizes, uint32_t nblocks, uint32_t starts, int on_device,
                            uint32_t* LFpowers, uint32_t* nLF, uint32_t* freqs, bwtc_cuda_stats* stats);
/* Streaming form of the same pipeline (the look-ahead driver of a compressor: read block, submit, keep reading; entropy-code
 * block i as soon as bwtc_cuda_pipeline_wait(i) returns).  submit queues ONE block (block contract, in/out as above; LFpowers:
 * 256 words, *nLF and freqs[256] written/incremented when the block completes; stats may be NULL) and returns at once with a
 * ticket; the pointers must stay valid until the block has been waited for.  Queued small blocks of equal size are still
 * batched into one device-side sort.  wait blocks (sleeping, not spinning) until that block is done and returns 0 or its
 * negative error (message: bwtc_cuda_pipeline_error).  Each ticket must be waited for exactly once. */
int  bwtc_cuda_pipeline_submit(bwtc_cuda_pipeline* p, const uint8_t* in, uint8_t* out, uint32_t n, uint32_t starts,
                               int on_device, uint32_t* LFpowers, uint32_t* nLF, uint32_t* freqs,
                               bwtc_cuda_stats* stats, uint64_t* ticket);
int  bwtc_cuda_pipeline_wait(bwtc_cuda_pipeline* p, uint64_t ticket);
/* Streaming inverse: queue ONE block (block contract of bwtc_cuda_inverse_block: in holds the n transformed bytes, the
 * original n bytes land in out, which may alias in; device memory when on_device != 0; eob = LFpowers[0] of the forward
 * transform; stats may be NULL) and return at once with a ticket of the same sequence as bwtc_cuda_pipeline_submit's; wait
 * for it with bwtc_cuda_pipeline_wait.  Queued inverse blocks of equal size are inverted as one device-side problem;
 * forward and inverse blocks are never grouped together.  An error is reported through every ticket of the group it
 * happened in, except BWTC_CUDA_ECORRUPT: only the ticket of a corrupt block returns it (its out buffer is untouched), the
 * other blocks of its group complete normally. */
int  bwtc_cuda_pipeline_submit_inverse(bwtc_cuda_pipeline* p, const uint8_t* in, uint8_t* out, uint32_t n, uint32_t eob,
                                       int on_device, bwtc_cuda_stats* stats, uint64_t* ticket);
/* submit + run statistics (filled when the block completes; such a block is transformed on its own, not in a batch).
 * in and out may differ (out-of-place host block).  runs->count is BWTC_CUDA_RUNS_OVERFLOW from this call on, and stays so
 * unless the block succeeds with at most runs->capacity runs. */
int  bwtc_cuda_pipeline_submit_runs(bwtc_cuda_pipeline* p, const uint8_t* in, uint8_t* out, uint32_t n, uint32_t starts,
                                    uint32_t* LFpowers, uint32_t* nLF, uint32_t* freqs, bwtc_cuda_runs* runs, uint64_t* ticket);
/* Device-side timing of whatever the pipeline's streams execute between the two calls: begin records
 * an event every context stream waits on; end joins all context streams and returns elapsed ms
 * (CUDA events, all streams of this pipeline), or a negative error. */
int   bwtc_cuda_pipeline_timing_begin(bwtc_cuda_pipeline* p);
float bwtc_cuda_pipeline_timing_end(bwtc_cuda_pipeline* p);

#ifdef __cplusplus
}
#endif
#endif /* BWTC_CUDA_H_ */
