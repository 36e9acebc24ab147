// Row statistics of float64 rows: the same 12 statistics, order and definitions as
// b200_rowstats (SURVEY.md App. B: population std, MAD about the mean, lower median,
// top-K / adjusted split), for the reference run under torch.set_default_dtype(float64).
//
// Order statistics are exact: the six-level select of select64.cuh (shared with the
// growth summaries) on the order-preserving key of the fp64 bit pattern resolves the
// four target ranks of rowstats.cu together:
//   j=0 med_all = (n-1)/2        j=1 thr     = n-K      (smallest of the top)
//   j=2 med_top = n-K+(K-1)/2    j=3 med_adj = (n-K-1)/2
// Moments are accumulated in fp64, about the group means (two passes per group).
// Eight streaming passes of 8 B per element:
//   pass 0      sum, counts of -inf / +inf / NaN, level-0 histogram
//   pass 1      level-1 histograms, |w - mean| and (w - mean)^2 of all
//   passes 2-5  level-2..5 histograms (after pass 5 thr is known exactly)
//   pass 6      sums / counts of the elements above and below thr (the ties of thr
//               are split between top and adj by count)
//   pass 7      deviations of top / adj about their own means
// Between passes a one-block-per-row resolve kernel extends the prefixes (one warp per
// target) or forms the means.  Single GPU only: no exchange phases.
#include "select64.cuh"

namespace b200 {

constexpr int R64_NT = 4;          // target ranks
constexpr int R64_THREADS = 256;
constexpr int R64_PASSES = 8;

struct RowWS64 {
  double sum_all, absdev_all, sqdev_all;
  double sum_gt, sum_lt, absdev_gt, sqdev_gt, absdev_lt, sqdev_lt;
  long long cnt_gt, cnt_lt, n_ninf, n_pinf, n_nan;
  long long hist[R64_NT][GBINS];   // level 0 uses hist[0] only
  long long rank[R64_NT];
  unsigned long long prefix[R64_NT];
  double mean_all, mean_top, mean_adj;
  double value[R64_NT];
};
static_assert(sizeof(RowWS64) % 8 == 0, "8-byte words");

// grid = (slices, rows)
template <int PASS>
__global__ void __launch_bounds__(R64_THREADS)
rowstats_f64_pass_kernel(const double* __restrict__ values, int64_t n, int64_t ld, RowWS64* __restrict__ ws) {
  extern __shared__ unsigned int r64_hist[];
  __shared__ double red_d[32];
  __shared__ long long red_i[32];
  constexpr bool SELECT = PASS < GLEVELS;
  constexpr int NH = PASS == 0 ? 1 : SELECT ? R64_NT : 0;
  const double* __restrict__ v = values + (int64_t)blockIdx.y * ld;
  RowWS64* w = ws + blockIdx.y;
  for (int i = threadIdx.x; i < NH * GBINS; i += R64_THREADS) r64_hist[i] = 0;
  unsigned long long pfx[R64_NT] = {};
  if (SELECT && PASS > 0) select64_prefixes<(SELECT ? PASS : 1), R64_NT>(w->prefix, pfx);
  const double mean_a = PASS == 1 ? w->mean_all : 0.0;
  const double mean_t = PASS == 7 ? w->mean_top : 0.0, mean_j = PASS == 7 ? w->mean_adj : 0.0;
  const unsigned long long thr_key = PASS >= GLEVELS ? w->prefix[1] : 0ull;   // the full key of thr
  __syncthreads();

  double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  long long c0 = 0, c1 = 0, c2 = 0;
  auto process = [&](double x) {
    const unsigned long long k = double_key(x);
    if (PASS == 0) {
      a0 += x;
      if (k == ~0ull) ++c2;
      else if (x == __longlong_as_double(0x7ff0000000000000LL)) ++c1;
      else if (x == -__longlong_as_double(0x7ff0000000000000LL)) ++c0;
    } else if (PASS == 1) {
      const double d = x - mean_a;
      a0 += fabs(d);
      a1 += d * d;
    } else if (PASS == 6) {
      if (k > thr_key) { a0 += x; ++c0; }
      else if (k < thr_key) { a1 += x; ++c1; }
    } else if (PASS == 7) {
      if (k > thr_key) { const double d = x - mean_t; a0 += fabs(d); a1 += d * d; }
      else if (k < thr_key) { const double d = x - mean_j; a2 += fabs(d); a3 += d * d; }
    }
    if (SELECT) select64_count<(SELECT ? PASS : 0), R64_NT>(k, pfx, r64_hist);
  };
  // four independent loads per thread in flight before the first is used (growth.cu)
  constexpr int U = 4;
  const int64_t stride = (int64_t)gridDim.x * R64_THREADS * U;
  for (int64_t base = (int64_t)blockIdx.x * R64_THREADS * U + threadIdx.x; base < n; base += stride) {
    double x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = base + (int64_t)u * R64_THREADS;
      x[u] = i < n ? __ldcs(v + i) : 0.0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (base + (int64_t)u * R64_THREADS < n) process(x[u]);
  }

  if (PASS == 0) {
    const double s = block_sum(a0, red_d);
    const long long ni = block_sum(c0, red_i), pi = block_sum(c1, red_i), nn = block_sum(c2, red_i);
    if (threadIdx.x == 0) {
      atomicAdd(&w->sum_all, s);
      if (ni) atomicAdd((unsigned long long*)&w->n_ninf, (unsigned long long)ni);
      if (pi) atomicAdd((unsigned long long*)&w->n_pinf, (unsigned long long)pi);
      if (nn) atomicAdd((unsigned long long*)&w->n_nan, (unsigned long long)nn);
    }
  } else if (PASS == 1) {
    const double s0 = block_sum(a0, red_d), s1 = block_sum(a1, red_d);
    if (threadIdx.x == 0) { atomicAdd(&w->absdev_all, s0); atomicAdd(&w->sqdev_all, s1); }
  } else if (PASS == 6) {
    const double s0 = block_sum(a0, red_d), s1 = block_sum(a1, red_d);
    const long long n0 = block_sum(c0, red_i), n1 = block_sum(c1, red_i);
    if (threadIdx.x == 0) {
      atomicAdd(&w->sum_gt, s0); atomicAdd(&w->sum_lt, s1);
      atomicAdd((unsigned long long*)&w->cnt_gt, (unsigned long long)n0);
      atomicAdd((unsigned long long*)&w->cnt_lt, (unsigned long long)n1);
    }
  } else if (PASS == 7) {
    const double s0 = block_sum(a0, red_d), s1 = block_sum(a1, red_d);
    const double s2 = block_sum(a2, red_d), s3 = block_sum(a3, red_d);
    if (threadIdx.x == 0) {
      atomicAdd(&w->absdev_gt, s0); atomicAdd(&w->sqdev_gt, s1);
      atomicAdd(&w->absdev_lt, s2); atomicAdd(&w->sqdev_lt, s3);
    }
  }
  if (NH > 0) {
    __syncthreads();
    for (int i = threadIdx.x; i < NH * GBINS; i += R64_THREADS) {
      const unsigned int c = r64_hist[i];
      if (c) atomicAdd((unsigned long long*)(&w->hist[0][0] + i), (unsigned long long)c);
    }
  }
}

// One block of 128 threads per row, after pass `step`.
__global__ void __launch_bounds__(128)
rowstats_f64_resolve_kernel(RowWS64* __restrict__ ws, int step, int64_t n, int64_t K, double* __restrict__ stats) {
  RowWS64* w = ws + blockIdx.x;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  if (step < GLEVELS) {
    // warp j resolves target j
    const int j = threadIdx.x >> 5;
    const long long first = j == 0 ? (n - 1) / 2 : j == 1 ? n - K : j == 2 ? n - K + (K - 1) / 2 : (n - K - 1) / 2;
    const long long* h = step == 0 ? w->hist[0] : w->hist[j];
    const long long rank = step == 0 ? first : w->rank[j];
    if (select64_resolve(h, step, rank, &w->prefix[j], &w->rank[j]) && step == GLEVELS - 1)
      w->value[j] = key_double(w->prefix[j]);
    __syncthreads();
    for (int i = threadIdx.x; i < R64_NT * GBINS; i += 128) (&w->hist[0][0])[i] = 0;
    if (step == 0 && threadIdx.x == 0) w->mean_all = w->sum_all / (double)n;
    return;
  }
  if (threadIdx.x != 0) return;
  const double thr = w->value[1];
  const long long n_eq = n - w->cnt_gt - w->cnt_lt;
  const long long tt = K - w->cnt_gt, ta = n_eq - tt;   // ties of thr in the top / adj group
  if (step == 6) {
    // a tie share of zero must not contribute 0 * inf
    w->mean_top = (w->sum_gt + (tt > 0 ? (double)tt * thr : 0.0)) / (double)K;
    w->mean_adj = n > K ? (w->sum_lt + (ta > 0 ? (double)ta * thr : 0.0)) / (double)(n - K) : qnan;
    return;
  }
  const double dt = thr - w->mean_top, da = thr - w->mean_adj;
  const double abs_top = w->absdev_gt + (tt > 0 ? (double)tt * fabs(dt) : 0.0);
  const double sq_top = w->sqdev_gt + (tt > 0 ? (double)tt * dt * dt : 0.0);
  const double abs_adj = w->absdev_lt + (ta > 0 ? (double)ta * fabs(da) : 0.0);
  const double sq_adj = w->sqdev_lt + (ta > 0 ? (double)ta * da * da : 0.0);
  double* s = stats + (int64_t)blockIdx.x * 12;
  s[0] = w->mean_all; s[1] = w->mean_top; s[2] = w->mean_adj;
  s[3] = w->absdev_all / (double)n; s[4] = abs_top / (double)K; s[5] = abs_adj / (double)(n - K);
  s[6] = sqrt(w->sqdev_all / (double)n); s[7] = sqrt(sq_top / (double)K); s[8] = sqrt(sq_adj / (double)(n - K));
  s[9] = w->value[0]; s[10] = w->value[2]; s[11] = w->value[3];
  // torch semantics, as rowstats.cu: a non-finite member makes std_mean's mean / std (hence MAD) nan, except
  // that a one-element group's mean is the element itself; a NaN member makes the median nan.  NaN sorts
  // greatest, -inf least.
  const long long ninf = w->n_ninf, nan = w->n_nan, hi = w->n_pinf + nan;
  const bool nonfinite[3] = {hi + ninf > 0, hi > 0 || ninf > n - K, hi > K || ninf > 0};
  const bool has_nan[3] = {nan > 0, nan > 0, nan > K};
  const long long size[3] = {n, K, n - K};
  const double single[3] = {w->value[0], w->value[1], w->value[3]};
  for (int g = 0; g < 3; ++g) {
    if (nonfinite[g]) { s[0 + g] = size[g] == 1 ? single[g] : qnan; s[3 + g] = qnan; s[6 + g] = qnan; }
    if (has_nan[g]) s[9 + g] = qnan;
  }
  if (n == K) { s[2] = qnan; s[5] = qnan; s[8] = qnan; s[11] = qnan; }   // empty adj group: torch gives nan
}

template <int PASS>
static void launch_r64_pass(dim3 grid, const double* v, int64_t n, int64_t ld, RowWS64* ws, cudaStream_t st) {
  constexpr int NH = PASS == 0 ? 1 : PASS < GLEVELS ? R64_NT : 0;
  rowstats_f64_pass_kernel<PASS><<<grid, R64_THREADS, (size_t)NH * GBINS * sizeof(unsigned int), st>>>(v, n, ld, ws);
}

}  // namespace b200

using namespace b200;

extern "C" int64_t b200_rowstats_f64_workspace_bytes(int64_t rows) {
  return rows < 0 ? 0 : rows * (int64_t)sizeof(RowWS64);
}

extern "C" int b200_rowstats_f64(const double* values, int64_t rows, int64_t n, int64_t ld, int64_t top,
                                 void* workspace, double* stats, void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(rows >= 0 && n >= 1, "rowstats_f64: need rows >= 0 and n >= 1");
  if (rows == 0) return 0;
  B200_REQUIRE(values != nullptr, "rowstats_f64: values is NULL");
  B200_REQUIRE(workspace != nullptr && stats != nullptr, "rowstats_f64: workspace/stats is NULL");
  B200_REQUIRE(top >= 1 && top <= n, "rowstats_f64: need 1 <= top <= n (top=%lld n=%lld)", (long long)top,
               (long long)n);
  B200_REQUIRE(ld >= n, "rowstats_f64: ld < n");
  if (rows > 65535) return set_error(B200_ELIMIT, "rowstats_f64: rows=%lld > 65535 per call", (long long)rows);
  cudaStream_t st = (cudaStream_t)stream;
  RowWS64* ws = (RowWS64*)workspace;
  const int64_t want = ((int64_t)sm_count() * 16 + rows - 1) / rows;
  const int64_t max_slices = (n + R64_THREADS * 16 - 1) / (R64_THREADS * 16);
  const int64_t slices = want < max_slices ? want : max_slices;
  const dim3 grid((unsigned)(slices < 1 ? 1 : slices), (unsigned)rows);
  B200_CUDA(cudaMemsetAsync(ws, 0, (size_t)rows * sizeof(RowWS64), st));
  for (int p = 0; p < R64_PASSES; ++p) {
    switch (p) {
      case 0: launch_r64_pass<0>(grid, values, n, ld, ws, st); break;
      case 1: launch_r64_pass<1>(grid, values, n, ld, ws, st); break;
      case 2: launch_r64_pass<2>(grid, values, n, ld, ws, st); break;
      case 3: launch_r64_pass<3>(grid, values, n, ld, ws, st); break;
      case 4: launch_r64_pass<4>(grid, values, n, ld, ws, st); break;
      case 5: launch_r64_pass<5>(grid, values, n, ld, ws, st); break;
      case 6: launch_r64_pass<6>(grid, values, n, ld, ws, st); break;
      case 7: launch_r64_pass<7>(grid, values, n, ld, ws, st); break;
    }
    rowstats_f64_resolve_kernel<<<(unsigned)rows, 128, 0, st>>>(ws, p, n, top, stats);
  }
  return check_cuda(cudaGetLastError(), "rowstats_f64 launch");
}
