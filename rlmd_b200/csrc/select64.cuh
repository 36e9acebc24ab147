// Exact order statistics of fp64 rows: a 6-level radix select (5 x 11 + 9 bits) on the
// order-preserving key of the fp64 bit pattern, several target ranks resolved together.
// Shared by the growth-rate summaries (growth.cu) and the fp64 row statistics
// (rowstats_f64.cu).  Per level, a pass kernel counts every key into the histogram of
// each target whose prefix it shares (select64_count), and one warp per target then
// walks that histogram (select64_resolve): the bin holding the target's remaining rank
// extends its prefix.  After the last level a prefix IS the key of the selected value.
#pragma once
#include "common.cuh"

namespace b200 {

constexpr int GBITS = 11, GBINS = 1 << GBITS;
constexpr int GLEVELS = 6;            // 11,11,11,11,11,9 bits

__host__ __device__ __forceinline__ unsigned long long double_key(double x) {
  unsigned long long b;
#ifdef __CUDA_ARCH__
  b = (unsigned long long)__double_as_longlong(x);
#else
  union { double d; unsigned long long u; } cv; cv.d = x; b = cv.u;
#endif
  if ((b & 0x7fffffffffffffffull) > 0x7ff0000000000000ull) return ~0ull;  // NaN sorts last (numpy / torch)
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_double(unsigned long long k) {
  if (k == ~0ull) return __longlong_as_double(0x7ff8000000000000LL);
  const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

__host__ __device__ __forceinline__ int level_shift(int level) { return level < 5 ? 64 - GBITS * (level + 1) : 0; }
__host__ __device__ __forceinline__ int level_bins(int level) { return level < 5 ? GBINS : 1 << 9; }

// The prefixes of the NT targets in the units select64_count compares at LEVEL (> 0).
template <int LEVEL, int NT>
__device__ __forceinline__ void select64_prefixes(const unsigned long long* prefix, unsigned long long (&pfx)[NT]) {
#pragma unroll
  for (int j = 0; j < NT; ++j) pfx[j] = prefix[j] >> (level_shift(LEVEL) + (LEVEL < 5 ? GBITS : 9));
}

// Key k into the shared-memory histograms of LEVEL: level 0 has one histogram of GBINS
// bins, every later level one per target (hist[j * GBINS + bin]).
template <int LEVEL, int NT>
__device__ __forceinline__ void select64_count(unsigned long long k, const unsigned long long (&pfx)[NT],
                                               unsigned int* hist) {
  constexpr int shift = LEVEL < 5 ? 64 - GBITS * (LEVEL + 1) : 0;
  if constexpr (LEVEL == 0) {
    atomicAdd(&hist[k >> shift], 1u);
  } else {
    const unsigned long long hi = k >> (shift + (LEVEL < 5 ? GBITS : 9));
    const unsigned int lo = (unsigned int)(k >> shift) & (unsigned int)(level_bins(LEVEL) - 1);
#pragma unroll
    for (int j = 0; j < NT; ++j)
      if (hi == pfx[j]) atomicAdd(&hist[j * GBINS + lo], 1u);
  }
}

// One warp (all 32 lanes call): the bin of histogram h (bins of `level`) that holds rank `want`
// extends *prefix (level 0: starts it) and *rank_out becomes the rank left inside that bin.
// Every lane sums a contiguous run of bins, a shuffle scan names the lane whose run holds
// the rank, that lane walks its run and stores.  Returns true on the storing lane.
__device__ __forceinline__ bool select64_resolve(const long long* h, int level, long long want,
                                                 unsigned long long* prefix, long long* rank_out) {
  const int lane = threadIdx.x & 31;
  const int bins = level_bins(level), shift = level_shift(level);
  const int per = bins / 32;   // 64 or 16
  long long local = 0;
  for (int i = 0; i < per; ++i) local += h[lane * per + i];
  long long incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long up = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += up;
  }
  const long long excl = incl - local;
  const long long total = __shfl_sync(0xffffffffu, incl, 31);
  const bool owner = (want >= excl && want < incl) || (lane == 31 && want >= total);
  if (owner) {
    long long r = want - excl;
    int b = lane * per;
    for (int i = 0; i < per; ++i) {
      const long long c = h[lane * per + i];
      if (r < c || i == per - 1) { b = lane * per + i; break; }
      r -= c;
    }
    const unsigned long long add = (unsigned long long)b << shift;
    *prefix = (level == 0 ? 0ull : *prefix) | add;
    *rank_out = r;
  }
  return owner;
}

}  // namespace b200
