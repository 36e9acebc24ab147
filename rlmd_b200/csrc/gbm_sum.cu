// GBM per-step series from the running log-return sum (gbm_smart_lev(..., method="sum")).
//
// Log wealth at leverage l after step t is log V0 + l S_t, S_t the investor's running sum of the
// log-returns, so at every step all leverages order the investors by S_t (ascending for l > 0,
// reversed for l < 0, all equal for l = 0).  One exact select on S per step gives the order
// statistics of every leverage; the moments take two passes over S with the wealth recomputed
// from S.  Nothing of size [G, steps, N] is written.
//
//   b200_gbm_sum_chunk : steps [t_begin, t_end) of x -> S rows [Tc, N] (fp32 x: GbmAcc's S, bit for
//                        bit the S of gbm_chunk_kernel; fp64 x: the sequential fp64 sum), state carried
//   b200_gbm_sum_stats : S rows [T, N] -> the 12 statistics of b200_rowstats (order, definitions) of
//                        every leverage at every row
//
// Statistics, per row (all launches cover every row of the call):
//   levels 0-5  select64 on the S keys at the four wealth ranks of rowstats.cu
//               j=0 (n-1)/2   j=1 n-K (thr)   j=2 n-K+(K-1)/2   j=3 (n-K-1)/2
//               and, when the grid holds an l < 0, their mirrors n-1-r (targets 4..7)
//   moments A   per leverage: sum of all, sums / counts above and below thr (ties split by count)
//   moments B   per leverage: |w - mean|, (w - mean)^2 about the all / top / adj means
// A moment block writes its partial sums to its own slot and the resolve kernel adds the slots in
// slice order, and the slices depend on n only: a row's statistics do not depend on how the
// horizon was chunked, nor on the run.
#include <cfloat>
#include <cmath>

#include "lev_kernels.cuh"
#include "select64.cuh"

namespace b200 {

constexpr int GS_THREADS = 256;
constexpr int GS_NT = 8;               // most targets: four ranks and their mirrors
constexpr int GS_GT = 4;               // leverages per moment block
constexpr int GS_SLICE = GS_THREADS * 16;
constexpr int GS_MAX_SLICES = 1024;
constexpr int GS_WORDS = 8;            // partial sums per (row, slice, leverage)

struct SumWS {
  long long hist[GS_NT][GBINS];        // level 0 uses hist[0] only
  long long rank[GS_NT];
  unsigned long long prefix[GS_NT];    // after level 5: the key of the selected S
  double mean_all[B200_MAX_GRID], mean_top[B200_MAX_GRID], mean_adj[B200_MAX_GRID];
  double sum[B200_MAX_GRID][7];        // moments A added over the slices
};
static_assert(sizeof(SumWS) % 8 == 0, "8-byte words");

struct SumLevs {
  double l[B200_MAX_GRID];
};

static int64_t sum_slices(int64_t n) {
  const int64_t s = (n + GS_SLICE - 1) / GS_SLICE;
  return s < 1 ? 1 : s > GS_MAX_SLICES ? GS_MAX_SLICES : s;
}

// gbm_wealth's expression (lev_sweep.cu): the chain's fp32 wealth bit for bit when f32
__device__ __forceinline__ double sum_wealth(double lv0, double l, double S, bool f32) {
  const double e = exp(lv0 + l * S);
  return f32 ? (double)(float)e : e;
}

// The S holding wealth rank target j of leverage l: S rank r for l >= 0, n-1-r (target j+4) for l < 0.
__device__ __forceinline__ double sum_target(const SumWS* w, double l, int j) {
  return key_double(w->prefix[(l < 0 ? 4 : 0) + j]);
}

// ----------------------------------------------------------------------------- S rows
template <bool F64>
__global__ void __launch_bounds__(128)
gbm_sum_chunk_kernel(const void* __restrict__ x, int64_t ld, int32_t t_begin, int32_t t_end, int64_t N,
                     double* __restrict__ state, double* __restrict__ S_out, int64_t ldS) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= N) return;
  if (F64) {
    const double* __restrict__ xr = (const double*)x + row * ld;
    double S = 0.0, mx = 0.0, mn = 0.0;
    if (t_begin > 0) { S = state[row]; mx = state[N + row]; mn = state[2 * N + row]; }
    for (int t = t_begin; t < t_end; ++t) {
      S += __ldg(xr + t);
      mx = fmax(mx, S);
      mn = fmin(mn, S);
      if (S_out != nullptr) S_out[(int64_t)(t - t_begin) * ldS + row] = S;
    }
    state[row] = S; state[N + row] = mx; state[2 * N + row] = mn;
    return;
  }
  const float* __restrict__ xr = (const float*)x + row * ld;
  GbmAcc acc;
  if (t_begin > 0) { acc.S = state[row]; acc.Smax = state[N + row]; acc.Smin = state[2 * N + row]; }
  for (int t = t_begin; t < t_end; ++t) {
    acc.step(__ldg(xr + t));
    if (S_out != nullptr) S_out[(int64_t)(t - t_begin) * ldS + row] = acc.S + (double)acc.p;   // gbm_chunk_kernel's S
    if ((t & 31) == 31) acc.fold();
  }
  acc.fold();
  state[row] = acc.S; state[N + row] = acc.Smax; state[2 * N + row] = acc.Smin;
}

// ----------------------------------------------------------------------------- select
// grid = (slices, rows)
template <int LEVEL, int NT>
__global__ void __launch_bounds__(GS_THREADS)
sum_select_kernel(const double* __restrict__ S, int64_t n, int64_t ld, SumWS* __restrict__ ws) {
  extern __shared__ unsigned int gs_hist[];
  constexpr int NH = LEVEL == 0 ? 1 : NT;
  const double* __restrict__ v = S + (int64_t)blockIdx.y * ld;
  SumWS* w = ws + blockIdx.y;
  for (int i = threadIdx.x; i < NH * GBINS; i += GS_THREADS) gs_hist[i] = 0;
  unsigned long long pfx[NT] = {};
  if constexpr (LEVEL > 0) select64_prefixes<LEVEL, NT>(w->prefix, pfx);
  __syncthreads();
  constexpr int U = 4;
  const int64_t stride = (int64_t)gridDim.x * GS_THREADS * U;
  for (int64_t base = (int64_t)blockIdx.x * GS_THREADS * U + threadIdx.x; base < n; base += stride) {
    double x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = base + (int64_t)u * GS_THREADS;
      x[u] = i < n ? __ldg(v + i) : 0.0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (base + (int64_t)u * GS_THREADS < n) select64_count<LEVEL, NT>(double_key(x[u]), pfx, gs_hist);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NH * GBINS; i += GS_THREADS) {
    const unsigned int c = gs_hist[i];
    if (c) atomicAdd((unsigned long long*)(&w->hist[0][0] + i), (unsigned long long)c);
  }
}

// ----------------------------------------------------------------------------- moments
// grid = (slices * gtiles, rows), the leverage tile fastest (the blocks of one slice read it from L2).
// PASS 0 partial words: sum, sum above thr, sum below thr, count above, count below, +inf, NaN.
// PASS 1: |d|, d^2 about the all / top (above thr) / adj (below thr) means.
template <int PASS, bool F32>
__global__ void __launch_bounds__(GS_THREADS)
sum_moment_kernel(const double* __restrict__ S, int64_t n, int64_t ld, const __grid_constant__ SumLevs L, int32_t G,
                  double lv0, int32_t gtiles, const SumWS* __restrict__ ws, double* __restrict__ part) {
  __shared__ double red_d[32];
  const int tile = blockIdx.x % gtiles;
  const int64_t slice = blockIdx.x / gtiles, slices = gridDim.x / gtiles;
  const int g0 = tile * GS_GT;
  const double* __restrict__ v = S + (int64_t)blockIdx.y * ld;
  const SumWS* w = ws + blockIdx.y;
  double l[GS_GT], thr[GS_GT], m0[GS_GT], m1[GS_GT], m2[GS_GT];
#pragma unroll
  for (int q = 0; q < GS_GT; ++q) {
    const int g = g0 + q < G ? g0 + q : G - 1;
    l[q] = L.l[g];
    thr[q] = sum_wealth(lv0, l[q], sum_target(w, l[q], 1), F32);
    m0[q] = PASS == 1 ? w->mean_all[g] : 0.0;
    m1[q] = PASS == 1 ? w->mean_top[g] : 0.0;
    m2[q] = PASS == 1 ? w->mean_adj[g] : 0.0;
  }
  double a[GS_GT][6] = {};
  int c[GS_GT][4] = {};
  const int64_t chunk = (n + slices - 1) / slices;
  const int64_t i0 = slice * chunk, i1 = i0 + chunk < n ? i0 + chunk : n;
  for (int64_t i = i0 + threadIdx.x; i < i1; i += GS_THREADS) {
    const double s = __ldg(v + i);
#pragma unroll
    for (int q = 0; q < GS_GT; ++q) {
      if (g0 + q >= G) continue;
      const double x = sum_wealth(lv0, l[q], s, F32);
      if (PASS == 0) {
        a[q][0] += x;
        if (x > thr[q]) { a[q][1] += x; ++c[q][0]; }
        else if (x < thr[q]) { a[q][2] += x; ++c[q][1]; }
        if (x == __longlong_as_double(0x7ff0000000000000LL)) ++c[q][2];
        else if (x != x) ++c[q][3];
      } else {
        const double d = x - m0[q];
        a[q][0] += fabs(d); a[q][1] += d * d;
        if (x > thr[q]) { const double e = x - m1[q]; a[q][2] += fabs(e); a[q][3] += e * e; }
        else if (x < thr[q]) { const double e = x - m2[q]; a[q][4] += fabs(e); a[q][5] += e * e; }
      }
    }
  }
  double* out = part + ((int64_t)blockIdx.y * slices + slice) * G * GS_WORDS;
#pragma unroll
  for (int q = 0; q < GS_GT; ++q) {
    if (g0 + q >= G) continue;     // uniform over the block
    constexpr int NW = PASS == 0 ? 7 : 6;
#pragma unroll
    for (int k = 0; k < NW; ++k) {
      double val;
      if (PASS == 0 && k >= 3) val = (double)c[q][k >= 3 ? k - 3 : 0];   // counts < 2^31: exact
      else val = a[q][k < 6 ? k : 0];
      const double r = block_sum(val, red_d);
      if (threadIdx.x == 0) out[(g0 + q) * GS_WORDS + k] = r;
    }
  }
}

// ----------------------------------------------------------------------------- resolve
// One block of 256 threads per row after select level `level`: warp j resolves target j, then the histograms
// that level used (level 0: one; later levels: one per target) are cleared for the next.
__global__ void __launch_bounds__(GS_THREADS)
sum_select_resolve_kernel(SumWS* __restrict__ ws, int level, int nt, int64_t n, int64_t K) {
  SumWS* w = ws + blockIdx.x;
  const int j = threadIdx.x >> 5;
  if (j < nt) {
    const long long ranks[4] = {(n - 1) / 2, n - K, n - K + (K - 1) / 2, (n - K - 1) / 2};
    const long long first = j < 4 ? ranks[j] : n - 1 - ranks[j - 4];
    const long long* h = level == 0 ? w->hist[0] : w->hist[j];
    select64_resolve(h, level, level == 0 ? first : w->rank[j], &w->prefix[j], &w->rank[j]);
  }
  __syncthreads();
  const int used = (level == 0 ? 1 : nt) * GBINS;
  for (int i = threadIdx.x; i < used; i += GS_THREADS) (&w->hist[0][0])[i] = 0;
}

// One block per row, one thread per leverage, after moment pass `pass`: 0 the means, 1 the 12 statistics.
__global__ void __launch_bounds__(B200_MAX_GRID)
sum_moment_resolve_kernel(SumWS* __restrict__ ws, const double* __restrict__ part, int64_t slices, int pass,
                          int64_t n, int64_t K, const __grid_constant__ SumLevs L, int32_t G, double lv0, bool f32,
                          int64_t rows, double* __restrict__ stats) {
  SumWS* w = ws + blockIdx.x;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  const int g = threadIdx.x;
  if (g >= G) return;
  const double* p = part + (int64_t)blockIdx.x * slices * G * GS_WORDS + g * GS_WORDS;
  const int nw = pass == 0 ? 7 : 6;
  double tot[7] = {0, 0, 0, 0, 0, 0, 0};
  for (int64_t s = 0; s < slices; ++s)
    for (int k = 0; k < nw; ++k) tot[k] += p[s * G * GS_WORDS + k];
  const double l = L.l[g];
  const double thr = sum_wealth(lv0, l, sum_target(w, l, 1), f32);
  if (pass == 0) {
    for (int k = 0; k < 7; ++k) w->sum[g][k] = tot[k];   // the non-finite counts (5, 6) are read after pass 1
    const long long cnt_gt = (long long)tot[3], cnt_lt = (long long)tot[4];
    const long long n_eq = n - cnt_gt - cnt_lt, tt = K - cnt_gt, ta = n_eq - tt;
    w->mean_all[g] = tot[0] / (double)n;
    // a tie share of zero must not contribute 0 * inf
    w->mean_top[g] = (tot[1] + (tt > 0 ? (double)tt * thr : 0.0)) / (double)K;
    w->mean_adj[g] = n > K ? (tot[2] + (ta > 0 ? (double)ta * thr : 0.0)) / (double)(n - K) : qnan;
    return;
  }
  const double* A = w->sum[g];
  const long long cnt_gt = (long long)A[3], cnt_lt = (long long)A[4];
  const long long pinf = (long long)A[5], nan = (long long)A[6];
  const long long n_eq = n - cnt_gt - cnt_lt, tt = K - cnt_gt, ta = n_eq - tt;
  const double mean_top = w->mean_top[g], mean_adj = w->mean_adj[g];
  const double dt = thr - mean_top, da = thr - mean_adj;
  const double abs_top = tot[2] + (tt > 0 ? (double)tt * fabs(dt) : 0.0);
  const double sq_top = tot[3] + (tt > 0 ? (double)tt * dt * dt : 0.0);
  const double abs_adj = tot[4] + (ta > 0 ? (double)ta * fabs(da) : 0.0);
  const double sq_adj = tot[5] + (ta > 0 ? (double)ta * da * da : 0.0);
  const double med = sum_wealth(lv0, l, sum_target(w, l, 0), f32);
  const double med_top = sum_wealth(lv0, l, sum_target(w, l, 2), f32);
  const double med_adj = sum_wealth(lv0, l, sum_target(w, l, 3), f32);
  double* s = stats + ((int64_t)g * rows + blockIdx.x) * 12;
  s[0] = w->mean_all[g]; s[1] = mean_top; s[2] = mean_adj;
  s[3] = tot[0] / (double)n; s[4] = abs_top / (double)K; s[5] = abs_adj / (double)(n - K);
  s[6] = sqrt(tot[1] / (double)n); s[7] = sqrt(sq_top / (double)K); s[8] = sqrt(sq_adj / (double)(n - K));
  s[9] = med; s[10] = med_top; s[11] = med_adj;
  // torch semantics, as rowstats.cu / rowstats_f64.cu (wealth is never -inf): a non-finite member makes
  // mean / MAD / std nan, except that a one-element group's mean is the element itself (fp32 rows: not for
  // the all group, as b200_rowstats); a NaN member makes the median nan; NaN and +inf sort greatest.
  const long long hi = pinf + nan;
  const bool nonfinite[3] = {hi > 0, hi > 0, hi > K};
  const bool has_nan[3] = {nan > 0, nan > 0, nan > K};
  const long long size[3] = {n, K, n - K};
  const double single[3] = {f32 ? qnan : med, thr, med_adj};
  for (int j = 0; j < 3; ++j) {
    if (nonfinite[j]) { s[0 + j] = size[j] == 1 ? single[j] : qnan; s[3 + j] = qnan; s[6 + j] = qnan; }
    if (has_nan[j]) s[9 + j] = qnan;
  }
  if (n == K) { s[2] = qnan; s[5] = qnan; s[8] = qnan; s[11] = qnan; }   // empty adj group: torch gives nan
}

template <int LEVEL, int NT>
static int launch_select(dim3 grid, const double* S, int64_t n, int64_t ld, SumWS* ws, cudaStream_t st) {
  constexpr int NH = LEVEL == 0 ? 1 : NT;
  constexpr size_t smem = (size_t)NH * GBINS * sizeof(unsigned int);
  if (smem > 48 * 1024)
    B200_CUDA(cudaFuncSetAttribute(sum_select_kernel<LEVEL, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem));
  sum_select_kernel<LEVEL, NT><<<grid, GS_THREADS, smem, st>>>(S, n, ld, ws);
  return 0;
}

template <int NT>
static int launch_level(int level, dim3 grid, const double* S, int64_t n, int64_t ld, SumWS* ws, cudaStream_t st) {
  switch (level) {
    case 0: return launch_select<0, NT>(grid, S, n, ld, ws, st);
    case 1: return launch_select<1, NT>(grid, S, n, ld, ws, st);
    case 2: return launch_select<2, NT>(grid, S, n, ld, ws, st);
    case 3: return launch_select<3, NT>(grid, S, n, ld, ws, st);
    case 4: return launch_select<4, NT>(grid, S, n, ld, ws, st);
    default: return launch_select<5, NT>(grid, S, n, ld, ws, st);
  }
}

}  // namespace b200

using namespace b200;

extern "C" int b200_gbm_sum_chunk(const void* x, int32_t x_f64, int64_t n_investors, int32_t horizon, int64_t ld_x,
                                  int32_t t_begin, int32_t t_end, double* state, double* S, int64_t ld_S,
                                  void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(n_investors >= 0 && horizon >= 1, "gbm_sum_chunk: need n_investors >= 0 and horizon >= 1");
  B200_REQUIRE(0 <= t_begin && t_begin < t_end && t_end <= horizon, "gbm_sum_chunk: need 0 <= t_begin < t_end <= horizon");
  B200_REQUIRE(x_f64 || (t_begin & 31) == 0, "gbm_sum_chunk: fp32 chunks start at a multiple of 32");
  if (n_investors == 0) return 0;
  B200_REQUIRE(x != nullptr && state != nullptr, "gbm_sum_chunk: NULL argument");
  B200_REQUIRE(ld_x >= horizon && (S == nullptr || ld_S >= n_investors),
               "gbm_sum_chunk: ld_x < horizon or ld_S < n_investors");
  const unsigned blocks = (unsigned)((n_investors + 127) / 128);
  cudaStream_t st = (cudaStream_t)stream;
  if (x_f64)
    gbm_sum_chunk_kernel<true><<<blocks, 128, 0, st>>>(x, ld_x, t_begin, t_end, n_investors, state, S, ld_S);
  else
    gbm_sum_chunk_kernel<false><<<blocks, 128, 0, st>>>(x, ld_x, t_begin, t_end, n_investors, state, S, ld_S);
  return check_cuda(cudaGetLastError(), "gbm_sum_chunk launch");
}

extern "C" int64_t b200_gbm_sum_stats_workspace_bytes(int64_t rows, int64_t n, int32_t n_grid) {
  if (rows < 0 || n < 1 || n_grid < 1) return 0;
  return rows * ((int64_t)sizeof(SumWS) + sum_slices(n) * n_grid * GS_WORDS * (int64_t)sizeof(double));
}

extern "C" int b200_gbm_sum_stats(const double* S, int64_t rows, int64_t n, int64_t ld, const double* lev_host,
                                  int32_t n_grid, double log_v0, int32_t round_f32, int64_t top, void* workspace,
                                  double* stats, void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(rows >= 0 && n >= 1, "gbm_sum_stats: need rows >= 0 and n >= 1");
  B200_REQUIRE(n_grid >= 1 && n_grid <= B200_MAX_GRID, "gbm_sum_stats: n_grid must be in 1..%d", B200_MAX_GRID);
  B200_REQUIRE(top >= 1 && top <= n, "gbm_sum_stats: need 1 <= top <= n (top=%lld n=%lld)", (long long)top,
               (long long)n);
  if (rows == 0) return 0;
  B200_REQUIRE(S != nullptr && lev_host != nullptr && workspace != nullptr && stats != nullptr,
               "gbm_sum_stats: NULL argument");
  B200_REQUIRE(ld >= n, "gbm_sum_stats: ld < n");
  if (rows > 65535) return set_error(B200_ELIMIT, "gbm_sum_stats: rows=%lld > 65535 per call", (long long)rows);
  SumLevs L;
  int nt = 4;
  for (int g = 0; g < B200_MAX_GRID; ++g) {
    L.l[g] = g < n_grid ? lev_host[g] : 0.0;
    if (g < n_grid && lev_host[g] < 0) nt = GS_NT;
  }
  cudaStream_t st = (cudaStream_t)stream;
  SumWS* ws = (SumWS*)workspace;
  double* part = (double*)((char*)workspace + rows * (int64_t)sizeof(SumWS));
  const int64_t slices = sum_slices(n);
  const int gtiles = (n_grid + GS_GT - 1) / GS_GT;
  const bool f32 = round_f32 != 0;
  B200_CUDA(cudaMemsetAsync(ws, 0, (size_t)rows * sizeof(SumWS), st));
  const dim3 sel_grid((unsigned)slices, (unsigned)rows);
  for (int level = 0; level < GLEVELS; ++level) {
    const int rc = nt == GS_NT ? launch_level<GS_NT>(level, sel_grid, S, n, ld, ws, st)
                               : launch_level<4>(level, sel_grid, S, n, ld, ws, st);
    if (rc) return rc;
    sum_select_resolve_kernel<<<(unsigned)rows, GS_THREADS, 0, st>>>(ws, level, nt, n, top);
  }
  const dim3 mom_grid((unsigned)(slices * gtiles), (unsigned)rows);
  for (int pass = 0; pass < 2; ++pass) {
    if (pass == 0 && f32)
      sum_moment_kernel<0, true><<<mom_grid, GS_THREADS, 0, st>>>(S, n, ld, L, n_grid, log_v0, gtiles, ws, part);
    else if (pass == 0)
      sum_moment_kernel<0, false><<<mom_grid, GS_THREADS, 0, st>>>(S, n, ld, L, n_grid, log_v0, gtiles, ws, part);
    else if (f32)
      sum_moment_kernel<1, true><<<mom_grid, GS_THREADS, 0, st>>>(S, n, ld, L, n_grid, log_v0, gtiles, ws, part);
    else
      sum_moment_kernel<1, false><<<mom_grid, GS_THREADS, 0, st>>>(S, n, ld, L, n_grid, log_v0, gtiles, ws, part);
    sum_moment_resolve_kernel<<<(unsigned)rows, B200_MAX_GRID, 0, st>>>(ws, part, slices, pass, n, top, L, n_grid,
                                                                        log_v0, f32, rows, stats);
  }
  return check_cuda(cudaGetLastError(), "gbm_sum_stats launch");
}
