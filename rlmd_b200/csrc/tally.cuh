// Tally of outcome-count tuples: the device-side table the discrete LOG count
// kernels feed from their epilogue.
//
// The final wealth of a discrete gamble (lev/lev_exp.py:83-87, :539-545,
// :1158-1168: value_0 * prod_t m[outcome_t]) depends on an investor's outcomes
// only through the counts (n_0, n_1[, n_2, n_3]) - so every investor with the
// same count tuple has the same wealth at EVERY leverage, and the reference's
// 12 summary statistics of [N] wealths (:89-104) are statistics of a few 1e4
// weighted bins (iid die rolls: n_k ~ Binomial(H, p_k), a blob of ~(10 sd)^(K-1)
// tuples).  The count kernel therefore ends with ONE hash-table insertion per
// investor row instead of G stores of data_T, and the statistics never read a
// [G,N] array at all (tally.cu).
//
// Table: open addressing, linear probing, 8-byte keys (~0 = empty) and 4-byte
// counts in separate arrays; key = n_1 | n_2 << 21 | n_3 << 42 (n_0 follows from
// the horizon; H < 2^21).  The table is sized for at most capacity / 2 distinct
// tuples; an overfull table shows as a long probe walk or as more tuples than the
// bin list holds, and either raises the overflow word (the statistics of that sweep
// are then flagged invalid - never silently wrong, never an unbounded walk).
#pragma once
#include "common.cuh"

namespace b200 {

constexpr unsigned long long TALLY_EMPTY = ~0ull;
constexpr int TALLY_COUNT_BITS = 21;                       // per outcome count
constexpr int64_t TALLY_MAX_HORIZON = (1 << TALLY_COUNT_BITS) - 1;

// header words (int64, device); 0..7 are the info words of include/rlmd_b200.h
enum {
  TH_NBINS = 0,     // distinct tuples of the last finalize
  TH_OVERFLOW = 1,  // != 0: a table or a bin list was too small; results invalid
  TH_BAD = 2,       // outcomes outside {0..K-1} met by an ingest kernel
  TH_TIMEOUT = 3,   // a peer's bins never arrived
  TH_MISMATCH = 4,  // sum of the bin counts != n_total at the last statistics call
  TH_RADIX = 5,     // grid points whose statistics took the radix route since the last finalize
  TH_TICKET = 9,    // last-block-done ticket of the compaction kernel
  TH_LISTPOS = 10,  // append cursor of the compaction kernel
  TH_CONCAT = 11,   // bins of all ranks before the merge removes duplicates
  TH_DEBUG = 16,    // 48 words of per-phase clock stamps (B200_TALLY_DEBUG builds)
  // Bounding box of (n_1, n_2) over the bin list, as 4 running maxima (identity 0):
  // TALLY_MAX_HORIZON - min n_1, max n_1, TALLY_MAX_HORIZON - min n_2, max n_2.
  // One atomic per block and word, never one per tuple.
  TH_BOX_ACC = 64,  // the single-GPU compaction's accumulators (published and cleared by its last block)
  TH_BOX = 68,      // the box of the list the statistics read
  TH_WORDS = 72
};

struct TallyDev {
  unsigned long long* keys;  // [mask + 1]; nullptr: no tally
  uint32_t* counts;          // [mask + 1]
  long long* header;         // [TH_WORDS]
  uint64_t mask;             // capacity - 1 (capacity a power of two)
};

__host__ __device__ __forceinline__ uint64_t tally_mix(uint64_t x) {   // murmur3 finalizer
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull;
  x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull;
  x ^= x >> 33;
  return x;
}

__host__ __device__ __forceinline__ uint64_t tally_key(int n1, int n2, int n3) {
  return (uint64_t)(uint32_t)n1 | ((uint64_t)(uint32_t)n2 << TALLY_COUNT_BITS) |
         ((uint64_t)(uint32_t)n3 << (2 * TALLY_COUNT_BITS));
}
__host__ __device__ __forceinline__ void tally_unkey(uint64_t key, int& n1, int& n2, int& n3) {
  n1 = (int)(key & TALLY_MAX_HORIZON);
  n2 = (int)((key >> TALLY_COUNT_BITS) & TALLY_MAX_HORIZON);
  n3 = (int)((key >> (2 * TALLY_COUNT_BITS)) & TALLY_MAX_HORIZON);
}

// counts[slot(key)] += add.  A slot only ever goes empty -> key inside one tally,
// so the plain (L2) read of the slot is safe: a stale "empty" just takes the CAS.
// No global fill counter (one address hit by every new tuple serialises the kernel's
// tail): a table kept at most half full by its sizing has clusters of a few slots,
// so a probe walk of TALLY_MAX_PROBE slots means it is overfull - that raises the
// overflow word (P(false alarm) ~ 0.82^256 per new tuple at load 1/2), and the
// compaction raises it when more tuples come out than the bin list holds.
constexpr int TALLY_MAX_PROBE = 256;
__device__ __forceinline__ void tally_insert(const TallyDev& t, uint64_t key, uint32_t add) {
  uint64_t slot = tally_mix(key) & t.mask;
  for (int probe = 0; probe < TALLY_MAX_PROBE; ++probe) {
    unsigned long long cur = __ldcg(t.keys + slot);
    if (cur == TALLY_EMPTY) {
      cur = atomicCAS(t.keys + slot, TALLY_EMPTY, (unsigned long long)key);
      if (cur == TALLY_EMPTY) cur = key;
    }
    if (cur == key) { atomicAdd(t.counts + slot, add); return; }
    slot = (slot + 1) & t.mask;
  }
  t.header[TH_OVERFLOW] = 1;
}

// host side (tally.cu): the device view of a caller's workspace
int tally_device_view(const ::b200_tally_plan* plan, void* workspace, int32_t horizon, TallyDev* out);

}  // namespace b200
