/*
 * rlmd_b200 - C ABI of the B200-native engine for rlmd's multiplicative
 * Monte-Carlo hot path (leverage sweeps, batched multiplicative env step,
 * replay-buffer n-step sampling).
 *
 * The reference (majidsina/rlmd) is pure Python and has NO plugin / FFI layer
 * (SURVEY.md section 8b): its boundary for this path is three sets of Python
 * signatures.  Each entry point below names the reference interface it sits
 * behind (file:line in the reference tree); rlmd_b200/{lev_exp,envs,
 * replay_torch}.py are the same-named Python shims that bind them with ctypes
 * (INTEGRATION.md shows the binding a maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the library never allocates or frees caller-visible memory;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - every call returns 0 or a negative B200_E* code; b200_last_error()
 *     returns the message of the last failing call on the calling thread;
 *   - no CPU fallback exists: without a CUDA device every compute entry point
 *     returns B200_ECUDA.
 */
#ifndef RLMD_B200_H
#define RLMD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_EINVAL (-1)  /* bad argument (message says which) */
#define B200_ECUDA (-2)   /* CUDA runtime / driver error */
#define B200_ELIMIT (-3)  /* size outside what the kernels support */

#define B200_MAX_PEERS 8   /* GPUs of one node that exchange over peer-mapped memory */

const char* b200_last_error(void);
int b200_version(void);
/* sm_count / cc_major / cc_minor of the current device */
int b200_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);

/* ------------------------------------------------------------------ *
 * Leverage sweep (K1)
 *
 * Sits behind lev/lev_exp.py: coin_fixed_final_lev :56, coin_smart_lev :128,
 * dice_* :508/:586, gbm_* :935/:1008, dice_sh_* :1121/:1209 - the per-leverage
 * loop `gambles = where(...); value = value_0 * prod / chain` (:83-87,
 * :167-175 and siblings) for the whole grid in one launch.
 * ------------------------------------------------------------------ */
enum {
  B200_LEV_DISCRETE = 0, /* coin / dice / dice_sh: factor table m[G][K]     */
  B200_LEV_GBM = 1       /* factor exp(l*x), x fp32 log-returns, lev[G]      */
};
enum {
  B200_SRC_STREAM = 0, /* pre-drawn outcomes [N,ld]: uint8 codes or fp32 x  */
  B200_SRC_PHILOX = 1  /* outcomes drawn on device, Philox4x32-10           */
};
enum {
  B200_MODE_CHAIN = 1, /* exact fp32 sequential product ((V0*m0)*m1)*...:
                          bit-identical to *_smart_lev's data_T (discrete)   */
  B200_MODE_LOG = 2    /* log-domain: integer outcome counts (discrete) or
                          fp64 sum of x (GBM); fp64 log-wealth               */
};

#define B200_MAX_GRID 64
#define B200_MAX_OUTCOMES 4

typedef struct b200_lev_desc {
  int64_t n_investors;     /* N: rows handled by this call (local shard)     */
  int64_t ld_outcomes;     /* row stride of `outcomes` in ELEMENTS (>= H)    */
  int64_t investor_offset; /* global id of row 0 (Philox counters, sharding) */
  int64_t ld_out;          /* row stride of data_T / log_w in elements; 0 = N
                              (lets a caller fill a column block of a wider
                              [G, N_total] array: host-pipelined / sharded runs) */
  uint64_t seed;           /* Philox key                                     */
  int32_t horizon;         /* H                                              */
  int32_t n_grid;          /* G <= B200_MAX_GRID                             */
  int32_t n_outcomes;      /* K in 2..4 (discrete); ignored for GBM          */
  int32_t kind;            /* B200_LEV_*                                     */
  int32_t source;          /* B200_SRC_*                                     */
  int32_t mode;            /* B200_MODE_*                                    */
  float value_0;           /* V0                                             */
  float log_mean;          /* GBM Philox: mean of x  (mu - sigma^2/2)        */
  float sigma;             /* GBM Philox: std of x                           */
  int32_t variant;         /* CHAIN kernel variant: 0 = library default,
                              1 FSEL, 2 LDS table, 3 FMA-pipe selection (all
                              bit-identical; exposed for benchmarking; 3 falls
                              back when a factor is not reproducible by one
                              fused multiply-add or K > 3)                    */
  uint32_t thresholds[B200_MAX_OUTCOMES]; /* discrete Philox: outcome =
                              #{k : draw >= thresholds[k]}, k < K-1, draw a
                              uniform uint32; thresholds ascending            */
  int32_t outcome_bits;    /* discrete STREAM outcomes: 0 or 8 = one uint8 code
                              per outcome; 2 = PACKED, four 2-bit codes per byte
                              (step t in byte t>>2, bits 2*(t&3)..+1), row
                              stride ld_outcomes in BYTES (>= ceil(H/4)).  A
                              fair die carries 1.25 bits per roll: the packed
                              array is a quarter of the HBM traffic of the LOG
                              sweep (the CHAIN kernels take uint8 codes);
                              1 = ONE bit per outcome (K = 2, the coin: step t in
                              byte t>>3, bit t&7; stride in bytes >= ceil(H/8))  */
  int32_t flags;           /* B200_LEV_FLAG_*                                    */
} b200_lev_desc;

/* GBM, LOG mode: data_T = fl32(exp(log wealth at H)) WITHOUT the running-extremes
 * saturation - the value `value_0 * exp(l x).prod(dim=1)` of gbm_fixed_final_lev
 * (lev/lev_exp.py:965-967: torch.prod multiplies in blocks, so it leaves the fp32
 * range only when the FINAL wealth does), whereas the default reproduces the
 * time-ordered chain of gbm_smart_lev (:1048-1055: inf / 0 for good once the
 * running wealth left the range). */
#define B200_LEV_FLAG_FINAL_ONLY 1
/* GBM, LOG mode: `log_w` receives double [3,N] = (S, max_t S_t, min_t S_t), S_t the running
 * sum of x - the leverage-INDEPENDENT state of an investor, from which every grid point's log
 * wealth (log V0 + l S), its fp32 saturation and hence its growth rate follow - instead of the
 * [G,N] log wealth: a tenth of the bytes at G = 10, and the growth-rate summaries of the whole
 * grid need ONE selection over S (b200_gbm_valid + b200_growth_summary on the row S). */
#define B200_LEV_FLAG_STATE_OUT 2
/* b200_tally_stats: the statistics run BESIDE another kernel (the next sweep, on another stream): the
 * select kernel then takes two CTAs per leverage instead of six - slower alone (more bins per CTA), but it
 * leaves the sweep its SMs (measured at 2 GPUs, statistics beside the next sweep: 0.448 against 0.469 ms per step). */
#define B200_LEV_FLAG_BESIDE_SWEEP 4
/* b200_tally_stats: every grid point takes the radix route (three histogram levels over the fp32 key)
 * instead of the log-wealth route - the route the kernel takes by itself for K = 4, non-finite log
 * factors, or a grid point whose log-wealth bins fail a check.  For comparing the two. */
#define B200_LEV_FLAG_RADIX_SELECT 8
/* b200_lev_tally on packed (2-bit / 1-bit) outcomes: the count kernel may start while the stream's previous
 * kernel still runs (programmatic dependent launch).  It streams the outcomes at once and waits for that kernel
 * to complete only before its first tally insertion or `counts` store, so the flag is for a stream whose
 * previous kernel writes nothing the sweep reads: FinalSweepPipeline sets it at depth 1, where that kernel is
 * the previous step's select, and the next sweep then runs on the SMs the statistics leave free.  The
 * environment variable B200_PDL=0 turns it (and the same launch mode of the compaction and the select) off. */
#define B200_LEV_FLAG_EARLY_START 16

/*
 * outcomes : STREAM: uint8 [N,ld] (discrete, codes < K; or packed 2-bit codes,
 *            see outcome_bits) or float [N,ld] (GBM); PHILOX: NULL.
 * factors_host : HOST pointer (the table is tiny and travels as a kernel
 *            parameter).  Discrete: float [G,K] row-major, computed by the
 *            caller with the reference's own fp32 expressions; GBM: float lev[G].
 * data_T   : float [G,N] wealth after step H-1, or NULL.
 *            CHAIN: the fp32 chain.  LOG: fl32(exp(log_w)) with the reference
 *            dtype's saturation (inf once the running wealth left fp32 range,
 *            0 once it underflowed: GBM tracks the running extremes).
 * log_w    : double [G,N] log wealth (LOG mode), or NULL.
 * counts   : int32 [N,K] occurrences of each outcome (discrete LOG), or NULL.
 */
int b200_lev_sweep(const b200_lev_desc* desc, const void* outcomes,
                   const float* factors_host, float* data_T, double* log_w,
                   int32_t* counts, void* stream);

/*
 * Per-step series (K2): steps [t_begin, t_end) of the sweep with the wealth
 * after EVERY step written out, for the per-step statistics of *_smart_lev
 * (lev/lev_exp.py:167-212 and siblings: `for lev: for t: value_t = ...; sort;
 * std_mean; median`).  The caller walks the horizon in chunks, runs
 * b200_rowstats over the [G * chunk] rows of `dump` and scatters the 12
 * statistics into data[G,13,H-1]; after the last chunk `state` holds data_T.
 *
 * state : discrete (CHAIN): float [G,N] wealth, in/out (ignored as input when
 *         t_begin == 0); GBM: double [5,N] = running sum of x, its max, its min,
 *         then the bit patterns of two 64-bit masks: bit g set once grid point g's
 *         wealth has overflowed / underflowed (sticky, the first one decides).
 * dump  : float [G, t_end - t_begin, N] or NULL (advance the state only).
 * t_begin must be a multiple of 4 (discrete Philox) / 32 (GBM).
 */
int b200_lev_chunk(const b200_lev_desc* desc, const void* outcomes,
                   const float* factors_host, int32_t t_begin, int32_t t_end,
                   void* state, float* dump, void* stream);

/* Materialises the outcomes a PHILOX sweep with `desc` consumes into
 * out[N,ld] (uint8 codes, packed 2-bit codes when desc->outcome_bits == 2 - then
 * ld_outcomes is in bytes and a multiple of 4 - or float x): lets a streamed run
 * and the CPU oracle see the identical pre-drawn array. */
int b200_lev_draw(const b200_lev_desc* desc, void* out, void* stream);

/* Wealth of a discrete sweep from the outcome COUNTS of a previous LOG sweep
 * (counts int32 [N,K], b200_lev_sweep's `counts` output): the leverage grid enters
 * the wealth only through log m[g][k], so a grid of any size - the 2-D leverage x
 * insurance-fraction grid of lev/dice_roll_sh.py's factor `1 + l r_k + (1-l) sh_k`
 * (lev/lev_exp.py:1160-1166) with both coefficients free - costs ONE pass over the
 * outcome array plus one call of this per tile of <= B200_MAX_GRID grid points.
 * desc: n_investors, n_grid, n_outcomes, value_0, ld_out as for b200_lev_sweep;
 * outputs bit-identical to the LOG sweep's. */
int b200_lev_from_counts(const b200_lev_desc* desc, const int32_t* counts,
                         const float* factors_host, float* data_T, double* log_w,
                         void* stream);

/* uint8 codes [N, ld_codes] -> packed 2-bit codes [N, ld_packed bytes]
 * (ld_packed >= ceil(H/4); codes are taken modulo 4, pad bits are written 0). */
int b200_lev_pack(const uint8_t* codes, int64_t n_investors, int32_t horizon,
                  int64_t ld_codes, uint8_t* packed, int64_t ld_packed, void* stream);
/* ... with the packed width chosen: bits = 2 (above) or 1 (the coin; codes taken modulo 2,
 * ld_packed >= ceil(H/8)). */
int b200_lev_pack_bits(const uint8_t* codes, int64_t n_investors, int32_t horizon,
                       int64_t ld_codes, uint8_t* packed, int64_t ld_packed, int32_t bits,
                       void* stream);

/* ------------------------------------------------------------------ *
 * Final-time statistics from outcome-count tuples ("tally")
 *
 * Sits behind {coin,dice,dice_sh}_fixed_final_lev (lev/lev_exp.py:56-125,
 * :508-583, :1121-1206): `value_T = value_0 * gambles.prod(dim=1)` followed by
 * the summary-statistic block (:89-104).  The product depends on an investor's
 * outcomes only through the counts (n_0 .. n_{K-1}), so investors with equal
 * count tuples have equal wealth at EVERY leverage: the count kernel ends with
 * one hash-table insertion per investor (no data_T), and the 12 statistics of
 * every leverage are exact weighted order statistics / fp64 moments over the
 * distinct tuples (a few 1e4 for iid rolls) - bit-identical medians and wealth
 * values to b200_lev_sweep(LOG) + b200_rowstats, which stay as the general path
 * (and the checker).  Across GPUs ONE exchange per sweep: the ranks' bin lists.
 *
 * Call sequence (all asynchronous on `stream`):
 *   b200_tally_reset                    once (and after an overflow)
 *   b200_lev_tally / b200_lev_ingest    one or more row blocks (chunks of a host array)
 *   b200_tally_finalize                 table -> distinct tuples (merged over ranks)
 *   b200_tally_stats                    any number of grids of <= grid_cap points
 * ------------------------------------------------------------------ */
typedef struct b200_tally_plan {
  int64_t rows_cap;   /* most investor rows tallied on THIS rank between two finalizes  */
  int64_t bins_cap;   /* most distinct count tuples after the merge (global); more
                         raises the overflow word instead of wrong statistics           */
  int32_t grid_cap;   /* most grid points per b200_tally_stats call, <= B200_MAX_GRID    */
  int32_t world;      /* ranks whose tallies are merged at finalize (1: this GPU only)   */
} b200_tally_plan;

/* bytes of device workspace / of the peer-mapped exchange buffer (0 when world == 1) */
int64_t b200_tally_workspace_bytes(const b200_tally_plan* plan);
int64_t b200_tally_exchange_bytes(const b200_tally_plan* plan);

/* Info words, int64 [B200_TALLY_INFO_WORDS] at the head of the workspace (device):
 *   0 distinct tuples of the last finalize      1 overflow (!= 0: statistics invalid)
 *   2 outcomes outside {0..K-1} met by b200_lev_ingest (dice: the reference would
 *     use such a value as the factor itself, lev/lev_exp.py:541; not supported)
 *   3 peer time-out (a rank's bins never arrived: statistics are NaN)
 *   4 sum of the bin counts seen by the last b200_tally_stats != n_total
 *   5 grid points whose statistics took the radix route (B200_LEV_FLAG_RADIX_SELECT)
 *     since the last finalize */
#define B200_TALLY_INFO_WORDS 8
int b200_tally_reset(const b200_tally_plan* plan, void* workspace, void* stream);

/* The discrete LOG count kernel of b200_lev_sweep with the tally as its sink:
 * desc / outcomes as for b200_lev_sweep (STREAM source: uint8 codes or packed
 * 2-bit codes; horizon < 2^21); counts int32 [N,K] or NULL. */
int b200_lev_tally(const b200_lev_desc* desc, const void* outcomes,
                   const b200_tally_plan* plan, void* workspace, int32_t* counts,
                   void* stream);

/* Reference-format outcomes -> engine format, counted on the way.
 * src: [N, ld_src] of `src_type` exactly as the reference scripts hold them -
 * coin: fp32 {0,1} (Bernoulli.sample, lev/coin_flip.py:160; code = (x == 1),
 * lev/lev_exp.py:85), dice: int64 {0,1,2} (Categorical.sample,
 * lev/dice_roll.py:147; cast to fp32 at lev/lev_exp.py:537) - or any of the
 * other types below.  Any combination of sinks (NULL = not wanted):
 *   codes   uint8 [N, ld_codes]   the CHAIN kernels' format (b200_lev_chunk)
 *   counts  int32 [N, K]
 *   tally   plan + workspace      the statistics' input (b200_tally_finalize)
 * One pass over src (8 B per outcome for int64: HBM-bound). */
enum { B200_DT_U8 = 0, B200_DT_I32 = 1, B200_DT_I64 = 2, B200_DT_F32 = 3, B200_DT_F64 = 4 };
int b200_lev_ingest(const void* src, int32_t src_type, int64_t n_investors, int32_t horizon,
                    int64_t ld_src, int32_t n_outcomes, uint8_t* codes, int64_t ld_codes,
                    int32_t* counts, const b200_tally_plan* plan, void* workspace,
                    void* stream);

/* Multi-GPU: rank r publishes its bins in exchange[r] (peer-mapped memory of
 * b200_tally_exchange_bytes, zeroed once) and every rank merges all of them in
 * rank order, keeping each tuple at its first occurrence - every rank ends with
 * the identical bin list, hence bit-identical statistics.  epoch = 1, 2, 3, ...:
 * one more per finalize, the same on every rank. */
typedef struct b200_tally_peers {
  void* exchange[B200_MAX_PEERS];
  int32_t world, rank;
  uint32_t epoch;
  uint32_t reserved;
} b200_tally_peers;

/* table -> distinct tuples (clears the table for the next sweep); peers NULL
 * when plan->world == 1.  phase = -1 runs everything; with world > 1, phase 0 =
 * publish (compaction into this rank's exchange buffer + its flag at every peer)
 * and phase 1 = merge (waits for the world's flags) can be issued separately - a
 * test that plays all ranks on ONE GPU publishes every rank before any merge, so
 * that no kernel ever waits for a kernel queued behind it. */
int b200_tally_finalize(const b200_tally_plan* plan, void* workspace,
                        const b200_tally_peers* peers, int32_t phase, void* stream);

/* The reference's 12 statistics (b200_rowstats order) of every grid point from the
 * finalized bins: desc supplies n_grid (<= grid_cap), n_outcomes, horizon, value_0;
 * factors_host float [G,K] as for b200_lev_sweep; n_total / top as for
 * b200_rowstats (2 <= n_total < 2^32).  stats double [G,12]. */
int b200_tally_stats(const b200_tally_plan* plan, void* workspace, const b200_lev_desc* desc,
                     const float* factors_host, int64_t n_total, int64_t top, double* stats,
                     void* stream);

/* ------------------------------------------------------------------ *
 * Row statistics (the reference's summary-statistic block)
 *
 * Sits behind the block inlined 13x in lev/lev_exp.py (e.g. :89-104,
 * :177-192): sort(descending); top = s[:K]; adj = s[K:]; std_mean
 * (population), lower median, MAD about the mean - for `rows` independent
 * vectors of length n in one call.  Exact order statistics by radix select on
 * the fp32 bit pattern (torch.sort order, NaN greatest).
 *
 * stats[r][12] (double), reference row order (lev/lev_exp.py:194-209):
 *   mean, mean_top, mean_adj, mad, mad_top, mad_adj,
 *   std, std_top, std_adj, med, med_top, med_adj.
 * ------------------------------------------------------------------ */
/* bytes of device workspace b200_rowstats needs for `rows` rows */
int64_t b200_rowstats_workspace_bytes(int64_t rows);

/* values: float [rows, ld] (row r at values + r*ld), n valid entries per row.
 * n_total / top describe the GLOBAL vector when the rows are investor shards
 * (multi-GPU): single-GPU callers pass n_total = n.
 * phase = -1 runs every pass back to back (single GPU).  phase = 0..4 runs
 * one pass; between passes a multi-GPU caller all-reduces (SUM) the
 * workspace's exchange region (see b200_rowstats_exchange) across ranks. */
int b200_rowstats(const float* values, int64_t rows, int64_t n, int64_t ld,
                  int64_t n_total, int64_t top, void* workspace, double* stats,
                  int32_t phase, void* stream);

/* Per-row regions of the workspace (viewed as [rows, out[4]] 8-byte words) that
 * must be summed across ranks after `phase`: out[0..1] = offset,count of the
 * int64 words, out[2..3] = offset,count of the double words, out[4] = words per
 * row. */
int b200_rowstats_exchange(int32_t phase, int64_t out[5]);

/* ------------------------------------------------------------------ *
 * Float64 leverage sweeps (the reference run under
 * torch.set_default_dtype(torch.float64): coin and GBM) - single GPU
 * ------------------------------------------------------------------ */
/* bytes of device workspace b200_rowstats_f64 needs for `rows` rows */
int64_t b200_rowstats_f64_workspace_bytes(int64_t rows);

/* The 12 statistics of b200_rowstats (same order and definitions) over double
 * rows: values double [rows, ld], n >= 1 entries per row, 1 <= top <= n (top == n:
 * the adj group is empty and its statistics are NaN, as torch's).  Exact order
 * statistics (select on the fp64 bit pattern, NaN greatest), fp64 moments.
 * stats double [rows, 12]. */
int b200_rowstats_f64(const double* values, int64_t rows, int64_t n, int64_t ld,
                      int64_t top, void* workspace, double* stats, void* stream);

/* Steps [t_begin, t_end) of the exact fp64 chain value <- value * m_t
 * (lev/lev_exp.py:160-212, :1042-1093).  desc: kind, n_investors, horizon,
 * ld_outcomes, n_grid (<= B200_MAX_GRID), n_outcomes as for b200_lev_chunk;
 * source must be B200_SRC_STREAM (value_0, seed and mode are not read).
 *   discrete: outcomes uint8 codes [N, ld], factors_host double [G,K], m = factors[g][code]
 *   GBM:      outcomes double x [N, ld],    factors_host double lev[G], m = exp(lev[g] * x)
 * state : double [G,N] wealth, in/out (value_0 everywhere before step 0).
 * dump  : double [G, t_end - t_begin, N] wealth after every step, or NULL. */
int b200_lev_chunk_f64(const b200_lev_desc* desc, const void* outcomes,
                       const double* factors_host, int32_t t_begin, int32_t t_end,
                       double* state, double* dump, void* stream);

/* ------------------------------------------------------------------ *
 * Per-step series of the coin from the up-move count lattice
 *
 * Sits behind coin_smart_lev (lev/lev_exp.py:128-237) when the caller opts in
 * (method="counts"): after step t an investor with k_t up-moves in steps 0..t
 * holds V0 u^k d^(t+1-k) at every leverage - monotone in k - so the 12
 * statistics of every leverage at step t follow from one integer histogram
 * hist[t][k].  The caller walks the horizon in chunks: count, then stats.
 * ------------------------------------------------------------------ */
/* One read of steps [t_begin, t_end) of the outcomes.
 * outcomes : outcome_bits = 8: uint8 codes [N, ld] (up = code & 1, the column of
 *            the factor table [G,2] = (down, up)); outcome_bits = 1: one bit per
 *            flip (b200_lev_pack_bits' layout; ld in bytes, a multiple of 4).
 * k_state  : int32 [N] up-moves in steps 0..t_begin-1 (ignored when t_begin == 0);
 *            on return, in steps 0..t_end-1.
 * hist     : int32 [t_end - t_begin, ld_hist], ld_hist >= horizon + 1, overwritten:
 *            row i = investors per k after step t_begin + i.
 * kmin/kmax: int32 [t_end - t_begin]: the occupied band of each row. */
int b200_coin_lattice_count(const void* outcomes, int64_t n_investors, int32_t horizon,
                            int64_t ld_outcomes, int32_t outcome_bits, int32_t t_begin,
                            int32_t t_end, int32_t* k_state, int32_t* hist, int64_t ld_hist,
                            int32_t* kmin, int32_t* kmax, void* stream);
/* The 12 statistics (b200_rowstats order and definitions, torch's non-finite rules,
 * 1 <= top <= n_investors; top == n_investors: the adj group is NaN) of every
 * leverage g and step t_begin + i from b200_coin_lattice_count's rows for those steps:
 * the wealth of bin k is exp(log_v0 + k log u + (t+1-k) log d) in fp64, rounded to
 * fp32 when round_f32; exact ranks by the cumulative counts, fp64 moments.
 * logs_host : HOST double [G,2] = (log d, log u) of each leverage (G <= B200_MAX_GRID).
 * stats     : double [G, n_steps, 12].
 * fails     : int32 [G], NOT cleared: += the steps at which leverage g fails the
 *             route rule - an extreme path (kmin[t] or kmax[t]) not strictly inside
 *             (FLT_MIN, FLT_MAX) (round_f32) / (DBL_MIN, DBL_MAX), with a margin of
 *             1e-3 in log space, or a log that is not finite.  The chain saturates
 *             path by path (inf and 0 absorb), the lattice does not: only a leverage
 *             that never fails may take the lattice's statistics. */
int b200_coin_lattice_stats(const int32_t* hist, int64_t ld_hist, const int32_t* kmin,
                            const int32_t* kmax, int32_t t_begin, int32_t n_steps,
                            const double* logs_host, int32_t n_grid, double log_v0,
                            int32_t round_f32, int64_t n_investors, int64_t top,
                            double* stats, int32_t* fails, void* stream);

/* ------------------------------------------------------------------ *
 * Per-step series of the three-outcome gamble from the count-tuple lattice
 *
 * Sits behind dice_smart_lev / dice_sh_smart_lev (lev/lev_exp.py:586-701,
 * :1209-1334) when the caller opts in (method="tuples"): after step t an
 * investor with a up-moves, b down-moves and c = t+1-a-b mid-moves holds
 * V0 u^a d^b m^c at every leverage, so the 12 statistics of every leverage at
 * step t follow from one integer histogram over the occupied (a, b) cells.
 * The caller walks the codes once for the bounds, lays every step's box out
 * flat, then walks them again in chunks: count, then stats.
 * outcomes: uint8 codes [N, ld] (0 up, 1 down, 2 mid: the columns of the factor
 * table [G,3]), unit inner stride, any ld >= horizon.
 * ab_state: int32 [2,N] = each investor's (a, b) over steps 0..t_begin-1 (ignored
 * when t_begin == 0); on return, over steps 0..t_end-1.
 * bounds  : int32 [4, ld_bounds] = amin, amax, bmin, bmax; column i = step
 *           t_begin + i.
 * ------------------------------------------------------------------ */
/* One read of steps [t_begin, t_end): the occupied bounds of every step. */
int b200_dice_lattice_bounds(const void* outcomes, int64_t n_investors, int32_t horizon,
                             int64_t ld_outcomes, int32_t t_begin, int32_t t_end,
                             int32_t* ab_state, int32_t* bounds, int64_t ld_bounds, void* stream);
/* One read of steps [t_begin, t_end) into hist int32 [hist_cells] (cleared first):
 * cell (a, b) of step t_begin + i is hist[offsets[i] + (a - amin) * (bmax - bmin + 1)
 * + (b - bmin)], bounds as b200_dice_lattice_bounds wrote them for those steps. */
int b200_dice_lattice_count(const void* outcomes, int64_t n_investors, int32_t horizon,
                            int64_t ld_outcomes, int32_t t_begin, int32_t t_end,
                            int32_t* ab_state, const int32_t* bounds, int64_t ld_bounds,
                            const int64_t* offsets, int32_t* hist, int64_t hist_cells,
                            void* stream);
/* The 12 statistics (b200_rowstats order and definitions, torch's non-finite rules,
 * 1 <= top <= n_investors; top == n_investors: the adj group is NaN) of every
 * leverage g and step t_begin + i from b200_dice_lattice_count's histogram of those
 * steps: the wealth of cell (a, b) is fl32(exp(log_v0 + a log u + b log d + c log m)),
 * evaluated in fp64 left to right; exact ranks by a select on that log value weighted
 * by the counts, fp64 moments summed in an order fixed by the step's box alone.
 * logs_host : HOST double [G,3] = (log u, log d, log m) of each leverage (G <= B200_MAX_GRID).
 * stats     : double [G, n_steps, 12].
 * fails     : int32 [G], NOT cleared: += the steps at which leverage g fails the
 *             route rule - the min or the max of the log value over the step's occupied
 *             cells not strictly inside (log FLT_MIN, log FLT_MAX) with a margin of 1e-3,
 *             a log that is not finite, or a select that cannot finish exactly (that
 *             step's statistics are then NaN).  Only a leverage that never fails may take
 *             the lattice's statistics. */
int b200_dice_lattice_stats(const int32_t* hist, const int32_t* bounds, int64_t ld_bounds,
                            const int64_t* offsets, int32_t t_begin, int32_t n_steps,
                            const double* logs_host, int32_t n_grid, double log_v0,
                            int64_t n_investors, int64_t top, double* stats, int32_t* fails,
                            void* stream);

/* ------------------------------------------------------------------ *
 * Per-step series of GBM from the running log-return sum
 *
 * Sits behind gbm_smart_lev (lev/lev_exp.py:1012-1120) when the caller opts in
 * (method="sum"): log wealth after step t is log V0 + l S_t at every leverage l,
 * S_t the running sum of the investor's log-returns, so one exact select on S_t
 * gives the order statistics of every leverage (the order reverses for l < 0)
 * and two passes over S_t its moments.  The caller walks the horizon in chunks:
 * S rows, then stats.
 * ------------------------------------------------------------------ */
/* Steps [t_begin, t_end) of x [N, ld_x] (x_f64 = 0: float, 1: double) into
 * S double [t_end - t_begin, ld_S] (row i = S after step t_begin + i).
 * state : double [3,N] = S, its running max and min (0 before step 0 counts),
 *         in/out (ignored as input when t_begin == 0).
 * float x: S is b200_lev_chunk's (32 steps in fp32 on the fp64 base, folded
 * when (t & 31) == 31), bit for bit; t_begin must be a multiple of 32.
 * double x: the sequential fp64 sum.  S may be NULL: advance the state only. */
int b200_gbm_sum_chunk(const void* x, int32_t x_f64, int64_t n_investors, int32_t horizon,
                       int64_t ld_x, int32_t t_begin, int32_t t_end, double* state, double* S,
                       int64_t ld_S, void* stream);
/* bytes of device workspace b200_gbm_sum_stats needs */
int64_t b200_gbm_sum_stats_workspace_bytes(int64_t rows, int64_t n, int32_t n_grid);
/* The 12 statistics (b200_rowstats order and definitions, torch's non-finite rules,
 * 1 <= top <= n; top == n: the adj group is NaN) of the wealth
 * w = exp(log_v0 + l * S) (rounded to fp32 when round_f32: gbm_smart_lev's chain
 * wealth bit for bit) of every leverage l and every row of S double [rows, ld].
 * Exact order statistics (select on S at the ranks and, for a grid with an l < 0,
 * their mirrors), fp64 moments; the same statistics however the rows are chunked.
 * lev_host : HOST double [n_grid] (n_grid <= B200_MAX_GRID).
 * stats    : double [n_grid, rows, 12]. */
int b200_gbm_sum_stats(const double* S, int64_t rows, int64_t n, int64_t ld,
                       const double* lev_host, int32_t n_grid, double log_v0,
                       int32_t round_f32, int64_t top, void* workspace, double* stats,
                       void* stream);

/* ------------------------------------------------------------------ *
 * Batched multiplicative environment step (K4)
 *
 * Sits behind the gym.Env classes of envs/coin_flip_envs.py (Coin_Inv{A,B,C}
 * :150-233,:290-379,:436-538), envs/dice_roll_envs.py, envs/gbm_envs.py
 * (:147-212,:304-323,:449-474) and envs/dice_roll_sh_envs.py (:160-235,
 * :290-365,:420-502,:557-645): `step(action) -> (next_state, reward,
 * [done, learn_done], risk)` and `reset()`, for n_envs independent copies in
 * lock-step; the done flags are tools/env_resources.py:26-137.  All fp64.
 * ------------------------------------------------------------------ */
enum { B200_ENV_COIN = 0, B200_ENV_DICE = 1, B200_ENV_GBM = 2, B200_ENV_DICE_SH = 3 };
enum { B200_INV_A = 0, B200_INV_B = 1, B200_INV_C = 2, B200_INV_INSURED = 3 };
#define B200_ENV_MAX_GAMBLES 8

typedef struct b200_env_desc {
  int32_t family;      /* B200_ENV_*                                          */
  int32_t investor;    /* B200_INV_* (INSURED: dice_sh only)                  */
  int32_t n_gambles;   /* simultaneous identical gambles (dice_sh: 1)         */
  int32_t stop_abs;    /* 1: stop-loss = |a0| (Coin_InvB, coin_flip_envs.py:308),
                          0: (a0 + eps1) / 2 (every other class)               */
  double max_value, initial_value, min_value;      /* 1e18, 1e4, 100            */
  double max_abs_action, min_reward, min_return;   /* eps1, eps2, eps3          */
  double max_return, min_weight, lev_factor;       /* 1e10, eps4, eta           */
  double returns[3];     /* coin: (up, down, -); dice: (up, down, mid)          */
  double probs[3];
  double sh_returns[3];  /* safe haven (up, down, mid), already clamped         */
  double i_lev_factor, sh_lev_factor;
  double log_mean, vol;  /* GBM: r ~ N(log_mean, vol)                           */
  uint64_t seed;         /* Philox key when returns are drawn on the device     */
} b200_env_desc;

/* state / action / risk vector lengths of the class `desc` describes */
int b200_menv_dims(const b200_env_desc* desc, int32_t* state_dim,
                   int32_t* action_dim, int32_t* risk_dim);

/* wealth [E], time [E] (per-env step counter, starts at 1), state [E,S] or NULL;
 * mask [E] bytes or NULL (= reset every env). */
int b200_menv_reset(const b200_env_desc* desc, int64_t n_envs, double* wealth,
                    int32_t* time, double* state, const uint8_t* mask, void* stream);

/* action [E,A]; returns_in [E,n_gambles] injected returns (dice_sh: the die
 * return, [E]) or NULL = draw on the device (Philox, `draw_index` must differ
 * for every call); next_state [E,S], reward [E], done [E,2] bytes
 * (done, learn_done), risk [E,R].  wealth / time are updated in place. */
int b200_menv_step(const b200_env_desc* desc, int64_t n_envs, double* wealth,
                   int32_t* time, const double* action, const double* returns_in,
                   uint64_t draw_index, double* next_state, double* reward,
                   uint8_t* done, double* risk, void* stream);

/* ------------------------------------------------------------------ *
 * Replay buffer (K5 gather / n-step return, K6 append)
 *
 * Sits behind tools/replay_torch.py ReplayBufferTorch (and its NumPy twin
 * tools/replay.py ReplayBuffer): __init__ :57-115, store_exp :167-197 with
 * _episode_history :117-165, sample_exp :360-412 with _construct_history
 * :199-247 and the multi-step return :273-358.  The caller owns every buffer
 * (the Python shim keeps them as the same-named torch tensors).
 * ------------------------------------------------------------------ */
#define B200_REPLAY_MAX_STEPS 64

typedef struct b200_replay_desc {
  int64_t mem_size;           /* slots (tools/replay_torch.py:79-82), < 2^31    */
  int32_t state_dim;          /* sum(input_dims)                                 */
  int32_t action_dim;         /* num_actions                                     */
  float* state_memory;        /* [mem_size, state_dim]                           */
  float* action_memory;       /* [mem_size, action_dim]                          */
  float* reward_memory;       /* [mem_size]                                      */
  float* next_state_memory;   /* [mem_size, state_dim]                           */
  uint8_t* terminal_memory;   /* [mem_size] 0/1                                  */
  int32_t* episode_start;     /* [mem_size] first slot of the slot's episode     */
  int64_t* header;            /* [8]: mem_idx, finished episodes, first / last
                                 terminal slot, first slot of the running episode;
                                 words 5..7: scratch of b200_replay_store (zero between calls) */
} b200_replay_desc;

/* zeroes the header, the terminal flags and episode_start (the reference's
 * T.empty leaves terminal_memory uninitialised, :98-100; its first-episode
 * branch :147 only works when that memory happens to be zero) */
int b200_replay_reset(const b200_replay_desc* desc, void* stream);

/* Appends `count` transitions in order, as `count` calls of store_exp would
 * (slot = (position + k) % mem_size; reward = fl32(max(reward, reward_floor)),
 * :189) and maintains episode_start / the header (_episode_history :117-165).
 * state [count,S], action [count,A], reward [count], next_state [count,S]:
 * double when is_f64 (the envs' dtype) else float; done [count] bytes.
 * position = mem_idx before the call, or -1 = take it from the device header
 * (no host round trip).  The multi-step bookkeeping assumes the append-only
 * regime the reference asserts (buffer >= n_cumsteps). */
int b200_replay_store(const b200_replay_desc* desc, const void* state, const void* action,
                      const void* reward, const void* next_state, const uint8_t* done,
                      int64_t count, int32_t is_f64, int64_t position, double reward_floor,
                      void* stream);

/* One transition from HOST memory - store_exp(state, action, reward,
 * next_state, done) as the training loop calls it (:167): the row travels as
 * a kernel parameter, so the call is one launch and no copy.
 * B200_ELIMIT when 2*state_dim + action_dim + 1 > 480. */
int b200_replay_store_host(const b200_replay_desc* desc, const double* state_host,
                           const double* action_host, double reward,
                           const double* next_state_host, int32_t done, int64_t position,
                           double reward_floor, void* stream);

/* n_batches mini-batches of `batch` samples in one call (sample_exp :360-412
 * is n_batches = 1).
 * idx      : int64 [n_batches*batch] slots to sample (the reference's `batch`,
 *            :383 - the parity path), or NULL = draw `batch` DISTINCT uniform
 *            slots per mini-batch on the device (Philox4x32-10 keyed by seed /
 *            draw_index, rejection of duplicates in a shared-memory set;
 *            batch <= 8192) and report them in out_idx.
 * filled   : min(mem_idx, mem_size) (:382), or -1 = from the device header.
 * multi_steps n in 1..64; gamma_pow_host: HOST float[n], fl32(gamma**t).
 * additive : 1 = sum of discounted rewards (dynamics "A"), 0 = product.
 * outputs  : out_state [.,S] (n = 1: state_memory[idx]; n > 1: the history's
 *            next_state at its first used step, :309), out_action [.,A],
 *            out_reward [.], out_next_state [.,S] = next_state_memory[idx],
 *            out_done [.] bytes, out_eff [.] int64 effective length (:336-345).
 *            A slot outside [0, filled) yields zeros and out_eff = 0. */
int b200_replay_sample(const b200_replay_desc* desc, const int64_t* idx, int64_t n_batches,
                       int32_t batch, int64_t filled, int32_t multi_steps,
                       const float* gamma_pow_host, int32_t additive, uint64_t seed,
                       uint64_t draw_index, int64_t* out_idx, float* out_state,
                       float* out_action, float* out_reward, float* out_next_state,
                       uint8_t* out_done, int64_t* out_eff, void* stream);

/* b200_replay_sample with nothing taken from the host at call time: the slots are always drawn on
 * the device, `filled` comes from the device header and the draw index from `counter` (device
 * int64 [2]: [0] the draw index, advanced by the call; [1] internal, zero-initialised).  The whole call can therefore be captured in a CUDA graph
 * once and replayed - one sample_exp per training step for the cost of a graph launch instead of
 * seven output allocations and a foreign-function call (tools/replay_torch.py:360-412 is called
 * once per learner step, algos/algo_sac.py:238-298). */
int b200_replay_sample_counted(const b200_replay_desc* desc, int64_t n_batches, int32_t batch,
                               int32_t multi_steps, const float* gamma_pow_host, int32_t additive,
                               uint64_t seed, int64_t* counter, int64_t* out_idx, float* out_state,
                               float* out_action, float* out_reward, float* out_next_state,
                               uint8_t* out_done, int64_t* out_eff, void* stream);

/* ------------------------------------------------------------------ *
 * Fused collector and evaluation rollouts (SURVEY.md section 8f row 2)
 *
 * Replaces the inner loop of scripts/rl_multiplicative.py:185-273
 *   next_state, reward, env_done, risk = env.step(action)
 *   agent.store_transistion(state, action, reward, next_state, learn_done)
 *   state = next_state      # env.reset() after a done step
 * for `n_envs` environments at once, and tools/eval_episodes.py:233-262 (the
 * n_eval constant-action episodes of eval_multiplicative).  Environment e
 * appends to lane e of the replay memory: its j-th transition sits at slot
 * j*n_envs + e (slot-major, so the appends of one step are contiguous rows),
 * with its own 8-word header at replay.header + 8*e, i.e. every lane is a
 * reference ReplayBufferTorch of lane_len slots (n_envs = 1: the reference's
 * single stream).  The step / sample counters that key the Philox draws live in
 * device memory (`counter`, int64[2]), so step + sample can be captured in a
 * CUDA graph and replayed without host work.
 * ------------------------------------------------------------------ */
typedef struct b200_collect_desc {
  b200_env_desc env;
  b200_replay_desc replay;  /* mem_size >= n_envs*lane_len; header int64 [n_envs, 8] */
  int64_t n_envs;
  int64_t lane_len;
  double reward_floor;      /* r_abs_zero, or -inf (tools/replay_torch.py:189)      */
} b200_collect_desc;

/* wealth [E], time [E], cur_state [E,S] (the observation the agent reads),
 * counter int64 [2] on the device; zeroes every lane header and the counters. */
int b200_collect_reset(const b200_collect_desc* desc, double* wealth, int32_t* time,
                       double* cur_state, int64_t* counter, void* stream);

/* One env step + append per environment.  action [E,A] double on the device;
 * returns_in [E,n_gambles] or NULL = Philox draws keyed by counter[0]; optional
 * outputs reward [E], done [E,2] bytes, risk [E,R] (NULL = not wanted).
 * cur_state becomes next_state, or the reset state after a done step. */
int b200_collect_step(const b200_collect_desc* desc, double* wealth, int32_t* time,
                      double* cur_state, const double* action, const double* returns_in,
                      int64_t* counter, double* reward, uint8_t* done, double* risk,
                      void* stream);

/* b200_replay_sample over the lanes: idx = slots (local*n_envs + lane) or NULL
 * = n_batches x batch distinct draws over the filled part of all lanes, keyed by
 * (seed, counter[1]); outputs as b200_replay_sample. */
int b200_collect_sample(const b200_collect_desc* desc, const int64_t* idx, int64_t n_batches,
                        int32_t batch, int32_t multi_steps, const float* gamma_pow_host,
                        int32_t additive, uint64_t seed, int64_t* counter, int64_t* out_idx,
                        float* out_state, float* out_action, float* out_reward,
                        float* out_next_state, uint8_t* out_done, int64_t* out_eff,
                        void* stream);

/* n_episodes evaluation episodes, one constant action [A] each (action
 * [n_episodes, A]), from the reset state until done or max_steps steps.
 * returns_in [max_steps, n_episodes, n_gambles] or NULL = Philox draws with
 * draw index draw_base + step (the stream b200_menv_step consumes with the same
 * seed and draw_index).  reward [n], steps int32 [n], risk [n,R] of the last
 * step taken; last_state [n,S] or NULL. */
int b200_menv_rollout(const b200_env_desc* desc, int64_t n_episodes, const double* action,
                      const double* returns_in, uint64_t draw_base, int32_t max_steps,
                      double* reward, int32_t* steps, double* risk, double* last_state,
                      void* stream);

/* ------------------------------------------------------------------ *
 * Market environments (SURVEY.md section 8f row 4)
 *
 * Sits behind envs/market_envs.py Market_Inv{A,B,C}_{D1,Dx}: reset(assets)
 * :204-222 / :684-703 and step(action, next_assets) :133-202, :283-358,
 * :440-528, :611-682, :765-841, :924-1013, with market_dones
 * (tools/env_resources.py:140-200).  The wealth update of the multiplicative
 * envs fed by historical prices: returns are next_assets / assets - 1 with
 * `assets` the prices handed to reset() (the reference never advances them).
 * ------------------------------------------------------------------ */
#define B200_MARKET_MAX_ASSETS 128

typedef struct b200_market_desc {
  int32_t investor;     /* B200_INV_A / _B / _C                                   */
  int32_t n_assets;     /* 1..128                                                 */
  int32_t obs_days;     /* 1 = the _D1 classes; > 1 = _Dx (state holds the history) */
  int32_t time_length;  /* step count that ends an episode (_Dx: the caller passes
                           time_length - obs_days + 1, envs/market_envs.py:581)    */
  double max_value, initial_value, min_value;      /* 1e34, 1e4, 100              */
  double max_abs_action, min_reward, min_return;   /* 0.99, 1e-3, -0.9            */
  double max_return, min_weight, lev_factor;       /* 1e10, 1e-5, 3               */
} b200_market_desc;

/* S = 4 + obs_days*n_assets, A = investor + n_assets, R as the reference's risk */
int b200_market_dims(const b200_market_desc* desc, int32_t* state_dim, int32_t* action_dim,
                     int32_t* risk_dim);

/* assets_in [E, obs_days*n_assets] (observed_market_state of step 0) is copied to
 * the env-owned `assets` [E, W]; wealth [E], time [E]; state [E,S] or NULL; mask
 * [E] bytes or NULL = every env. */
int b200_market_reset(const b200_market_desc* desc, int64_t n_envs, double* wealth,
                      int32_t* time, const double* assets_in, double* assets, double* state,
                      const uint8_t* mask, void* stream);

/* action [E,A], next_assets [E,W]; next_state [E,S], reward [E], done [E,2] bytes
 * (done, learn_done), risk [E,R].  wealth / time are updated in place. */
int b200_market_step(const b200_market_desc* desc, int64_t n_envs, double* wealth,
                     int32_t* time, const double* assets, const double* action,
                     const double* next_assets, double* next_state, double* reward,
                     uint8_t* done, double* risk, void* stream);

/* ------------------------------------------------------------------ *
 * Multi-GPU statistics exchange (SURVEY.md section 8e)
 *
 * After phase p of b200_rowstats / b200_growth_summary every rank must sum, per
 * row, the integer words [int_offset, +int_count) and the double words
 * [dbl_offset, +dbl_count) of its workspace with its peers (the *_exchange calls
 * name them).  pack gathers both regions of all rows into ONE contiguous fp64
 * buffer staging[rows, int_count + dbl_count] (counts are < 2^53: exact), the
 * caller all-reduces it (one NCCL call per phase), unpack scatters it back.
 * ------------------------------------------------------------------ */
/* The same exchange WITHOUT a collective library, for the GPUs of one node: the
 * ranks' workspaces (and small flag blocks) live in memory every process has
 * mapped (CUDA IPC / torch symmetric memory).  Rows are owned round-robin
 * (row % world).  After each pass a rank pushes every row's partial sums into the
 * staging area of the row's owner (posted stores over NVLink) and flags its peers;
 * the owner waits for the world's flags, sums its rows' partials (ranks in the same
 * order) into shared memory, resolves them there and stores the few resolved words
 * - finally the 12 statistics - into every rank's workspace: a histogram crosses
 * NVLink once, and all ranks end with bit-identical statistics.
 *   stage[r]     : rank r's staging area, b200_rowstats_stage_bytes(rows, world) bytes:
 *                  [source rank][stage_rows][words]; alternates with the workspaces
 *   workspace[r] : rank r's rowstats workspace as mapped HERE (>= workspace_bytes(rows))
 *   flags[r]     : rank r's flag block, uint32 [B200_PEER_FLAG_WORDS], zeroed once;
 *                  word B200_PEER_FLAG_ERROR_WORD of the own block is set when a peer's
 *                  flag did not arrive within ~60 s (the statistics are then NaN)
 *   epoch        : 1, 2, 3, ... - one more per call, the same on every rank; successive
 *                  calls must alternate between two workspaces (a peer may still be
 *                  reading the previous call's sums)
 * Runs the whole statistic block (all passes) on `stream`. */
#define B200_PEER_FLAG_ERROR_WORD (B200_MAX_PEERS * 8)
#define B200_PEER_FLAG_WORDS 128
typedef struct b200_peer_set {
  void* workspace[B200_MAX_PEERS];
  uint32_t* flags[B200_MAX_PEERS];
  void* stage[B200_MAX_PEERS];   /* rank r's staging area as mapped HERE (b200_rowstats_stage_bytes) */
  int64_t stage_rows;            /* owned rows a staging area holds per source rank: >= ceil(rows / world) */
  int32_t world, rank;
  uint32_t epoch;
  uint32_t reserved;
} b200_peer_set;
int64_t b200_rowstats_stage_bytes(int64_t rows, int32_t world);
int b200_rowstats_p2p(const float* values, int64_t rows, int64_t n, int64_t ld,
                      int64_t n_total, int64_t top, const b200_peer_set* peers,
                      double* stats, void* stream);

int b200_exchange_pack(const void* workspace, int64_t words_per_row, int64_t rows,
                       int64_t int_offset, int64_t int_count, int64_t dbl_offset,
                       int64_t dbl_count, double* staging, void* stream);
int b200_exchange_unpack(void* workspace, int64_t words_per_row, int64_t rows,
                         int64_t int_offset, int64_t int_count, int64_t dbl_offset,
                         int64_t dbl_count, const double* staging, void* stream);

/* ------------------------------------------------------------------ *
 * Growth-rate summaries (engine-added; SURVEY.md App. B)
 *
 * The reference forms the time-average growth rate only as the env reward
 * exp(log(W/W0)/t) (envs/coin_flip_envs.py:183-185) and summarises with mean /
 * median / 5th percentile, np.percentile(method="median_unbiased")
 * (tools/eval_episodes.py:276-315, plotting/plots_multiverse.py:167-169).
 * Per row of log_w (the LOG sweep's fp64 log wealth, one row per leverage):
 *   g_i = (log_w_i - log_v0) / horizon
 * out[r][6 + n_q] (double):
 *   0 valid runs (data_T finite and > 0: survived the reference's fp32 wealth;
 *     data_T NULL -> log_w finite), 1 mean g, 2 population std g,
 *   3 mean g over the valid runs, 4 min g, 5 max g,
 *   6.. the n_q (<= 3) quantiles, Hyndman-Fan type 8 = numpy "median_unbiased"
 *   (two equal neighbours, e.g. both -inf, give that value instead of numpy's nan).
 * Exact order statistics (radix select on the fp64 bit pattern).  phase = -1
 * runs everything; phase 0..6 one step each, a multi-GPU caller summing the
 * words named by b200_growth_exchange(phase) over ranks in between.
 * ------------------------------------------------------------------ */
int64_t b200_growth_workspace_bytes(int64_t rows);

/* GBM: per grid point, the runs that survive the reference's fp32 wealth - out double [G,2] =
 * (count, sum of S over them) - from the sweep's state [3,N] (B200_LEV_FLAG_STATE_OUT) and its
 * data_T [G, ld_T] (finite and > 0); data_T NULL: the wealth is re-formed from the state with
 * the sweep's own saturation rule (one exp per run and grid point).  `out` is overwritten. */
int b200_gbm_valid(const double* state, const float* data_T, int64_t n, int64_t ld_T,
                   const float* lev_host, int32_t n_grid, double log_v0, double* out, void* stream);

/* GBM: the growth-rate summaries of the whole grid, out double [G, 6 + n_q] in
 * b200_growth_summary's layout, from base_row = the b200_growth_summary row of S (log_v0 = 0,
 * horizon = 1; its quantile columns hold the quantiles the caller asked of S) and valid [G,2]
 * (b200_gbm_valid, summed over ranks): g = l S / H, so every column scales with l / H, and a row
 * with l < 0 takes S's mirrored quantile (type 8 is symmetric) and swaps min / max.
 * pick_pos / pick_neg : device int32 [n_q]: which quantile column of base_row output column q
 * reads for l >= 0 / l < 0. */
int b200_gbm_growth_assemble(const double* base_row, const double* valid, const float* lev_host,
                             int32_t n_grid, int32_t horizon, int32_t n_q, const int32_t* pick_pos,
                             const int32_t* pick_neg, double* out, void* stream);
int b200_growth_exchange(int32_t phase, int64_t out[5]);
int b200_growth_summary(const double* log_w, const float* data_T, int64_t rows, int64_t n,
                        int64_t ld, int64_t ld_T, int64_t n_total, double log_v0,
                        int32_t horizon, const double* quantiles_host, int32_t n_q,
                        void* workspace, double* out, int32_t phase, void* stream);

/* ------------------------------------------------------------------ *
 * State-dependent leverage sweeps (K3, "big brain")
 *
 * Sits behind lev/lev_exp.py coin_big_brain_lev :270-452 (with coin_optimal_lev
 * :240-267) and dice_big_brain_lev :741-932 (dice_optimal_lev :704-738): for
 * every (retention, stop-loss) grid point the chain
 *   lev = eta (1 - floor(V) / V);  V <- V (1 + lev g_t)
 * with the wealth after / leverage before every step written out for the
 * per-step statistics (b200_rowstats) of data[R,S,26,H-1].
 * ------------------------------------------------------------------ */
enum { B200_BB_COIN = 0, /* fp32 chain (lev/lev_exp.py:323-379)                  */
       B200_BB_DICE = 1  /* float64 wealth chain, mixed-precision leverage (:791) */ };
#define B200_BB_MAX_POINTS 128

typedef struct b200_bigbrain_desc {
  int64_t n_investors;   /* N (local shard)                                       */
  int64_t ld_outcomes;   /* row stride of the uint8 outcome codes                 */
  int32_t horizon;       /* H                                                     */
  int32_t n_points;      /* grid points of this call, <= B200_BB_MAX_POINTS       */
  int32_t kind;          /* B200_BB_*                                             */
  int32_t reserved;
  float value_0;         /* V0 (fp32 like the scripts' tensor)                    */
  float lev_factor32;    /* fl32(LEV_FACTOR)                                      */
  double lev_factor64;   /* LEV_FACTOR (a float64 0-dim tensor in the scripts)    */
  double returns[3];     /* return of outcome code 0,1,2 (coin: down, up, -;
                            dice: up, down, mid)                                  */
} b200_bigbrain_desc;

/*
 * Steps [s_begin, s_end) of the recurrence (step s consumes outcome column s;
 * step 0 is the initialisation with the scalar leverage lev0 and writes no dump).
 * stop_vmin_host / roll_host / lev0_host : HOST arrays [n_points]: fl32(stop*V0),
 *            the fp32 retention ratio, and the float64 leverage of step 0.
 * state    : float (coin) / double (dice) [2, n_points, N]: wealth then leverage;
 *            in/out (ignored as input when s_begin == 0).
 * dump     : float [n_points, s_end - max(s_begin,1), 2, N]: per step the leverage
 *            BEFORE the update (statistic rows 12..23 of column s-1) and the
 *            wealth AFTER it (rows 0..11); NULL = advance the state only.
 */
int b200_bigbrain_chunk(const b200_bigbrain_desc* desc, const uint8_t* outcomes,
                        const float* stop_vmin_host, const float* roll_host,
                        const double* lev0_host, int32_t s_begin, int32_t s_end, void* state,
                        float* dump, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RLMD_B200_H */
