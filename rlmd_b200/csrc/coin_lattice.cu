// Per-step series of a two-outcome gamble (the coin) from the up-move count lattice
// (coin_smart_lev(..., method="counts"); DESIGN.md section 6.9).
//
// After step t an investor with k up-moves in steps 0..t holds V0 u^k d^(t+1-k) at EVERY
// leverage, monotone in k, so the 12 statistics of every leverage at step t follow from one
// integer histogram hist[t][k] over the occupied band [kmin[t], kmax[t]]:
//   count : one read of the outcomes -> hist, kmin, kmax (and each investor's running k);
//   stats : per (leverage, step) a warp walks the band in ascending wealth order - exact ranks
//           from the cumulative counts, fp64 moments, the top / adj split by count.
//
// The count kernel keeps k in registers: a block owns 256 * R investors and walks the steps of
// the call in tiles of 32, accumulating a shared-memory histogram [32][CNT_W] of k relative to
// the block's smallest k at the tile's start, and flushes only the occupied part of it with one
// global atomic per non-zero bin.  A k that falls outside the window (a block whose investors
// spread over more than CNT_W - 33 up-moves) goes straight to the global histogram: correct at
// any spread, fast when the spread is that of iid flips.
#include <cfloat>
#include <climits>
#include <cmath>

#include "common.cuh"

namespace b200 {

constexpr int CNT_THREADS = 256;
constexpr int CNT_TT = 32;       // steps per tile: one 32-bit word of a 1-bit row
constexpr int CNT_W = 376;       // window of k per tile: 32 x 376 x 4 B = 47 KB of static shared memory

// 32 uint8 codes (4 per word) -> one bit each (code & 1), step b of the four in bit b
__device__ __forceinline__ uint32_t byte_bits(uint32_t w) { return ((w & 0x01010101u) * 0x01020408u) >> 24; }

// The outcome word of tile `tile` of row `row`: bit s = up-move at step 32 * tile + s, for the steps in
// [t_lo, t_hi) (other bits are whatever the row holds there and are never read).
template <int BITS>
__device__ __forceinline__ uint32_t tile_word(const uint8_t* __restrict__ row, int tile, int t_lo, int t_hi,
                                              bool aligned) {
  if (BITS == 1) return __ldg(reinterpret_cast<const uint32_t*>(row) + tile);
  const int t0 = tile * CNT_TT;
  uint32_t m = 0;
  if (aligned) {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      if (t0 + 16 * q >= t_hi) break;        // (ld is a multiple of 16 >= horizon: a started piece is in the row)
      const uint4 w = __ldg(reinterpret_cast<const uint4*>(row + t0 + 16 * q));
      m |= (byte_bits(w.x) | byte_bits(w.y) << 4 | byte_bits(w.z) << 8 | byte_bits(w.w) << 12) << (16 * q);
    }
  } else {
    for (int t = t_lo; t < t_hi; ++t) m |= (uint32_t)(__ldg(row + t) & 1u) << (t - t0);
  }
  return m;
}

template <int BITS, int R>
__global__ void __launch_bounds__(CNT_THREADS)
lattice_count_kernel(const uint8_t* __restrict__ outcomes, int64_t N, int64_t ld, bool aligned, int32_t t_begin,
                     int32_t t_end, int32_t* __restrict__ k_state, int32_t* __restrict__ hist, int64_t ld_hist) {
  __shared__ int32_t sh[CNT_TT * CNT_W];
  __shared__ int32_t red[2][CNT_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t i0 = (int64_t)blockIdx.x * CNT_THREADS * R + tid;
  int k[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t i = i0 + (int64_t)r * CNT_THREADS;
    k[r] = (i < N && t_begin > 0) ? k_state[i] : 0;
  }
  for (int j = tid; j < CNT_TT * CNT_W; j += CNT_THREADS) sh[j] = 0;

  for (int tile = t_begin / CNT_TT; tile * CNT_TT < t_end; ++tile) {
    const int t0 = tile * CNT_TT;
    const int t_lo = max(t_begin, t0), t_hi = min(t_end, t0 + CNT_TT);
    // the block's band at the tile's start: window base and the occupied width
    int lo = INT_MAX, hi = INT_MIN;
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (i0 + (int64_t)r * CNT_THREADS < N) { lo = min(lo, k[r]); hi = max(hi, k[r]); }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    if (lane == 0) { red[0][wid] = lo; red[1][wid] = hi; }
    __syncthreads();       // (also: the previous tile's flush is done with sh)
    lo = red[0][0]; hi = red[1][0];
#pragma unroll
    for (int w = 1; w < CNT_THREADS / 32; ++w) { lo = min(lo, red[0][w]); hi = max(hi, red[1][w]); }
    uint32_t m[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int64_t i = i0 + (int64_t)r * CNT_THREADS;
      m[r] = i < N ? tile_word<BITS>(outcomes + i * ld, tile, t_lo, t_hi, aligned) : 0u;
    }
    for (int t = t_lo; t < t_hi; ++t) {
      const int s = t - t0;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (i0 + (int64_t)r * CNT_THREADS >= N) continue;
        k[r] += (int)((m[r] >> s) & 1u);
        const int j = k[r] - lo;
        if (j < CNT_W) atomicAdd(sh + s * CNT_W + j, 1);
        else atomicAdd(hist + (int64_t)(t - t_begin) * ld_hist + k[r], 1);
      }
    }
    __syncthreads();
    // flush: row s holds k in [lo, hi + s + 1]
    for (int t = t_lo; t < t_hi; ++t) {
      const int s = t - t0;
      const int width = min(CNT_W, hi - lo + s + 2);
      int32_t* dst = hist + (int64_t)(t - t_begin) * ld_hist + lo;
      for (int j = tid; j < width; j += CNT_THREADS) {
        const int c = sh[s * CNT_W + j];
        if (c != 0) { atomicAdd(dst + j, c); sh[s * CNT_W + j] = 0; }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t i = i0 + (int64_t)r * CNT_THREADS;
    if (i < N) k_state[i] = k[r];
  }
}

// kmin / kmax of every histogram row: one warp per row (row i is step t_begin + i: bins 0 .. t + 1)
__global__ void __launch_bounds__(256)
lattice_band_kernel(const int32_t* __restrict__ hist, int64_t ld_hist, int32_t t_begin, int32_t n_steps,
                    int32_t* __restrict__ kmin, int32_t* __restrict__ kmax) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_steps) return;
  const int32_t* h = hist + (int64_t)row * ld_hist;
  const int bins = t_begin + row + 2;
  int lo = INT_MAX, hi = -1;
  for (int j = lane; j < bins; j += 32)
    if (h[j] != 0) { lo = min(lo, j); hi = max(hi, j); }
  lo = __reduce_min_sync(0xffffffffu, lo);
  hi = __reduce_max_sync(0xffffffffu, hi);
  if (lane == 0) { kmin[row] = lo; kmax[row] = hi; }
}

struct LatticeLogs {
  double lu[B200_MAX_GRID], ld[B200_MAX_GRID];    // log u, log d per leverage of this call
};

// exp(log V0 + k log u + (t+1-k) log d) in fp64 (the library is built with -fmad=false: the expression rounds
// as written, left to right), rounded to fp32 when the series is fp32
__device__ __forceinline__ double lattice_value(double lv0, double lu, double ld, int t, int k, bool f32) {
  const double v = exp(lv0 + (double)k * lu + (double)(t + 1 - k) * ld);
  return f32 ? (double)__double2float_rn(v) : v;
}

__device__ __forceinline__ long long warp_incl_scan(long long v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

// One warp per (leverage, step).  Wealth ascends with k when log u >= log d, else descends: position p of the
// walk is k = kmin + p or kmax - p, so the walk visits the values in ascending order.
__global__ void __launch_bounds__(256)
lattice_stats_kernel(const int32_t* __restrict__ hist, int64_t ld_hist, const int32_t* __restrict__ kmin,
                     const int32_t* __restrict__ kmax, int32_t t_begin, int32_t n_steps,
                     const __grid_constant__ LatticeLogs L, int32_t G, double lv0, bool f32, long long n, long long K,
                     double lw_lo, double lw_hi, double* __restrict__ stats, int32_t* __restrict__ fails) {
  const int64_t pair = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pair >= (int64_t)G * n_steps) return;
  const int g = (int)(pair / n_steps), row = (int)(pair % n_steps), t = t_begin + row;
  const double lu = L.lu[g], ld = L.ld[g];
  const int lo = kmin[row], hi = kmax[row];
  const int32_t* h = hist + (int64_t)row * ld_hist;
  double* s = stats + pair * 12;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);

  if (lane == 0) {   // route rule: both extreme paths strictly inside the dtype's normal range (margin in lw_lo/hi)
    const double a = lv0 + (double)lo * lu + (double)(t + 1 - lo) * ld;
    const double b = lv0 + (double)hi * lu + (double)(t + 1 - hi) * ld;
    if (!(fmin(a, b) > lw_lo && fmax(a, b) < lw_hi)) atomicAdd(fails + g, 1);
  }
  if (!isfinite(lu) || !isfinite(ld) || lo > hi) {
    if (lane < 12) s[lane] = qnan;
    return;
  }
  const bool asc = lu >= ld;
  const int bins = hi - lo + 1;
  const long long n_adj = n - K;
  const long long ranks[4] = {(n - 1) / 2, n - K, n - K + (K - 1) / 2, (n_adj - 1) / 2};
  const long long rank_ok[4] = {1, 1, 1, n_adj > 0};

  // pass 1: ranks, sums, non-finite members per group
  double med[4] = {0, 0, 0, 0}, sum[3] = {0, 0, 0};
  int inf_[3] = {0, 0, 0};
  long long base = 0;
  for (int p0 = 0; p0 < bins; p0 += 32) {
    const int p = p0 + lane;
    const int kk = asc ? lo + p : hi - p;
    const long long c = p < bins ? h[kk] : 0;
    const double v = c > 0 ? lattice_value(lv0, lu, ld, t, kk, f32) : 0.0;
    const long long after = base + warp_incl_scan(c, lane), before = after - c;
    const long long tc = c > 0 ? max(0LL, after - max(before, n - K)) : 0, ac = c - tc;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const unsigned hit = __ballot_sync(0xffffffffu, rank_ok[j] && c > 0 && before <= ranks[j] && ranks[j] < after);
      if (hit) med[j] = __shfl_sync(0xffffffffu, v, __ffs(hit) - 1);
    }
    if (c > 0) { sum[0] += (double)c * v; inf_[0] |= isinf(v); }
    if (tc > 0) { sum[1] += (double)tc * v; inf_[1] |= isinf(v); }
    if (ac > 0) { sum[2] += (double)ac * v; inf_[2] |= isinf(v); }
    base = __shfl_sync(0xffffffffu, after, 31);
  }
  double mean[3];
  const double size[3] = {(double)n, (double)K, (double)n_adj};
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    mean[j] = warp_sum(sum[j]) / size[j];
    inf_[j] = __any_sync(0xffffffffu, inf_[j]);
  }

  // pass 2: absolute and squared deviations about each group's mean
  double dev[3] = {0, 0, 0}, sq[3] = {0, 0, 0};
  base = 0;
  for (int p0 = 0; p0 < bins; p0 += 32) {
    const int p = p0 + lane;
    const int kk = asc ? lo + p : hi - p;
    const long long c = p < bins ? h[kk] : 0;
    const long long after = base + warp_incl_scan(c, lane), before = after - c;
    const long long tc = c > 0 ? max(0LL, after - max(before, n - K)) : 0, ac = c - tc;
    if (c > 0) {
      const double v = lattice_value(lv0, lu, ld, t, kk, f32);
      const double cnt[3] = {(double)c, (double)tc, (double)ac};
#pragma unroll
      for (int j = 0; j < 3; ++j)
        if (cnt[j] > 0) {
          const double e = v - mean[j];
          dev[j] += cnt[j] * fabs(e);
          sq[j] += cnt[j] * (e * e);
        }
    }
    base = __shfl_sync(0xffffffffu, after, 31);
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) { dev[j] = warp_sum(dev[j]); sq[j] = warp_sum(sq[j]); }

  if (lane == 0) {
    // torch semantics (as rowstats / the tally): a non-finite member makes mean / MAD / std nan, except that a
    // one-element group's mean is the element itself; an empty adj group is all nan
    const double single[3] = {med[0], med[1], med[3]};
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      s[0 + j] = mean[j];
      s[3 + j] = dev[j] / size[j];
      s[6 + j] = sqrt(sq[j] / size[j]);
      if (inf_[j]) { s[0 + j] = size[j] == 1 ? single[j] : qnan; s[3 + j] = qnan; s[6 + j] = qnan; }
    }
    s[9] = med[0]; s[10] = med[2]; s[11] = med[3];
    if (n_adj == 0) { s[2] = qnan; s[5] = qnan; s[8] = qnan; s[11] = qnan; }
  }
}

}  // namespace b200

using namespace b200;

extern "C" int b200_coin_lattice_count(const void* outcomes, int64_t n_investors, int32_t horizon, int64_t ld_outcomes,
                                       int32_t outcome_bits, int32_t t_begin, int32_t t_end, int32_t* k_state,
                                       int32_t* hist, int64_t ld_hist, int32_t* kmin, int32_t* kmax, void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(outcome_bits == 8 || outcome_bits == 1, "coin_lattice_count: outcome_bits must be 8 or 1");
  B200_REQUIRE(n_investors >= 1 && horizon >= 1, "coin_lattice_count: need n_investors >= 1 and horizon >= 1");
  B200_REQUIRE(n_investors <= INT_MAX, "coin_lattice_count: more than 2^31 - 1 investors per histogram bin");
  B200_REQUIRE(0 <= t_begin && t_begin < t_end && t_end <= horizon,
               "coin_lattice_count: need 0 <= t_begin < t_end <= horizon");
  B200_REQUIRE(ld_hist >= (int64_t)horizon + 1, "coin_lattice_count: ld_hist < horizon + 1");
  B200_REQUIRE(outcomes != nullptr && k_state != nullptr && hist != nullptr && kmin != nullptr && kmax != nullptr,
               "coin_lattice_count: NULL argument");
  const bool aligned = ((uintptr_t)outcomes & 15) == 0 && ld_outcomes % 16 == 0;
  if (outcome_bits == 1) {
    B200_REQUIRE(ld_outcomes >= ((int64_t)horizon + 7) / 8 && ld_outcomes % 4 == 0 && ((uintptr_t)outcomes & 3) == 0,
                 "coin_lattice_count: 1-bit rows need ld_outcomes >= ceil(horizon/8), a multiple of 4, and a 4-byte "
                 "aligned array");     // (then the 32-bit word holding the last step lies inside the row)
  } else {
    B200_REQUIRE(ld_outcomes >= horizon, "coin_lattice_count: ld_outcomes < horizon");
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int32_t steps = t_end - t_begin;
  B200_CUDA(cudaMemsetAsync(hist, 0, (size_t)steps * (size_t)ld_hist * sizeof(int32_t), st));
  // investors per thread: the fewest that still fit the grid into one wave of four blocks per SM
  const int64_t wave = 4LL * sm_count();
  int R = 1;
  while (R < 8 && (n_investors + (int64_t)CNT_THREADS * R - 1) / ((int64_t)CNT_THREADS * R) > wave) R *= 2;
  const unsigned blocks = (unsigned)((n_investors + (int64_t)CNT_THREADS * R - 1) / ((int64_t)CNT_THREADS * R));
  const uint8_t* oc = (const uint8_t*)outcomes;
#define B200_LATTICE_COUNT(BITS, RR)                                                                              \
  lattice_count_kernel<BITS, RR><<<blocks, CNT_THREADS, 0, st>>>(oc, n_investors, ld_outcomes, aligned, t_begin, \
                                                                 t_end, k_state, hist, ld_hist)
  if (outcome_bits == 1) {
    if (R == 1) B200_LATTICE_COUNT(1, 1); else if (R == 2) B200_LATTICE_COUNT(1, 2);
    else if (R == 4) B200_LATTICE_COUNT(1, 4); else B200_LATTICE_COUNT(1, 8);
  } else {
    if (R == 1) B200_LATTICE_COUNT(8, 1); else if (R == 2) B200_LATTICE_COUNT(8, 2);
    else if (R == 4) B200_LATTICE_COUNT(8, 4); else B200_LATTICE_COUNT(8, 8);
  }
#undef B200_LATTICE_COUNT
  B200_CUDA(cudaGetLastError());
  lattice_band_kernel<<<(unsigned)((steps + 7) / 8), 256, 0, st>>>(hist, ld_hist, t_begin, steps, kmin, kmax);
  return check_cuda(cudaGetLastError(), "coin_lattice_count launch");
}

extern "C" int b200_coin_lattice_stats(const int32_t* hist, int64_t ld_hist, const int32_t* kmin, const int32_t* kmax,
                                       int32_t t_begin, int32_t n_steps, const double* logs_host, int32_t n_grid,
                                       double log_v0, int32_t round_f32, int64_t n_investors, int64_t top,
                                       double* stats, int32_t* fails, void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(n_grid >= 1 && n_grid <= B200_MAX_GRID, "coin_lattice_stats: n_grid must be in 1..%d", B200_MAX_GRID);
  B200_REQUIRE(t_begin >= 0 && n_steps >= 1, "coin_lattice_stats: need t_begin >= 0 and n_steps >= 1");
  B200_REQUIRE(ld_hist >= (int64_t)t_begin + n_steps + 1, "coin_lattice_stats: ld_hist too small for the steps");
  B200_REQUIRE(n_investors >= 1 && top >= 1 && top <= n_investors, "coin_lattice_stats: need 1 <= top <= n_investors");
  B200_REQUIRE(hist != nullptr && kmin != nullptr && kmax != nullptr && logs_host != nullptr && stats != nullptr &&
               fails != nullptr, "coin_lattice_stats: NULL argument");
  LatticeLogs L;
  for (int g = 0; g < B200_MAX_GRID; ++g) {
    L.ld[g] = g < n_grid ? logs_host[2 * g] : 0.0;
    L.lu[g] = g < n_grid ? logs_host[2 * g + 1] : 0.0;
  }
  const double margin = 1e-3;
  const double lw_lo = round_f32 ? std::log((double)FLT_MIN) + margin : std::log(DBL_MIN) + margin;
  const double lw_hi = round_f32 ? std::log((double)FLT_MAX) - margin : std::log(DBL_MAX) - margin;
  const int64_t pairs = (int64_t)n_grid * n_steps;
  lattice_stats_kernel<<<(unsigned)((pairs + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      hist, ld_hist, kmin, kmax, t_begin, n_steps, L, n_grid, log_v0, round_f32 != 0, n_investors, top, lw_lo, lw_hi,
      stats, fails);
  return check_cuda(cudaGetLastError(), "coin_lattice_stats launch");
}
