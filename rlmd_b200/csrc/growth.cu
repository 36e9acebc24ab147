// Growth-rate summaries of a leverage sweep (the "time-average growth rate"
// reductions named by the north star; SURVEY.md App. B "engine-added summaries").
//
// The reference forms the time-average growth only as the env reward
// exp(log(W/W0)/t) (envs/coin_flip_envs.py:183-185) and summarises per-episode
// quantities with mean / median / 5th percentile, np.percentile(...,
// method="median_unbiased") (tools/eval_episodes.py:276-315; the leverage plots
// take the same percentile of data_T, plotting/plots_multiverse.py:167-169).
// Here, per leverage row of log_w [G,N] (fp64 log wealth of the LOG sweep):
//     g_i = (log_w_i - log V0) / H
//     valid   = #{i : data_T_i finite and > 0}  (runs that survived the
//               reference dtype: its fp32 wealth overflows / underflows silently)
//     mean, population std of g over all runs; mean of g over the valid runs;
//     min, max; up to three Hyndman-Fan type-8 quantiles (numpy "median_unbiased").
// Order statistics are exact: a 6-level radix select (5 x 11 + 9 bits) on the
// order-preserving key of the fp64 bit pattern resolves all eight target ranks
// (lower / upper neighbour of each quantile, min, max) together; g is monotone in
// log_w, so selecting on log_w selects g.  Six streaming passes of 8 B/element,
// every cross-block quantity an 8-byte workspace word (summed across ranks by a
// multi-GPU caller, like b200_rowstats).
#include "select64.cuh"

namespace b200 {

constexpr int GT = 8;                 // target ranks
constexpr int G_THREADS = 256;

struct GrowthWS {
  // doubles (exchange after pass 0: [0,2); after pass 1: [2,3))
  double sum_g, sum_g_valid, sqdev, pad_d[5];
  // integers (exchange after pass 0: cnt_valid)
  long long cnt_valid, pad_i[7];
  long long hist[GT][GBINS];          // level 0 uses hist[0] only
  // resolved
  long long rank[GT];
  unsigned long long prefix[GT];
  double mean;
  double value[GT];
  long long pad_r[7];
};
static_assert(sizeof(GrowthWS) % 8 == 0, "8-byte words");
constexpr int64_t GW_OFF_CNT = 8, GW_OFF_HIST = 16, GW_ROW_WORDS = sizeof(GrowthWS) / 8;

struct GrowthParams {
  long long rank[GT];   // ascending 0-based target ranks in the global vector
  double frac[3];       // interpolation weight of the upper neighbour per quantile
  double log_v0, h;
  int n_q;
};

// grid = (slices, rows)
template <int LEVEL>
__global__ void __launch_bounds__(G_THREADS)
growth_pass_kernel(const double* __restrict__ log_w, const float* __restrict__ data_T, int64_t n, int64_t ld,
                   int64_t ld_T, GrowthWS* __restrict__ ws, const __grid_constant__ GrowthParams p) {
  extern __shared__ unsigned int g_hist[];
  __shared__ double red_d[32];
  __shared__ long long red_i[32];
  const int64_t row = blockIdx.y;
  const double* __restrict__ v = log_w + row * ld;
  const float* __restrict__ w32 = data_T ? data_T + row * ld_T : nullptr;
  GrowthWS* w = ws + row;
  constexpr int NH = LEVEL == 0 ? 1 : GT;
  for (int i = threadIdx.x; i < NH * GBINS; i += G_THREADS) g_hist[i] = 0;
  unsigned long long pfx[GT];
  double mean = 0.0;
  if (LEVEL > 0) select64_prefixes<LEVEL, GT>(w->prefix, pfx);
  if (LEVEL == 1) mean = w->mean;
  __syncthreads();

  double a0 = 0, a1 = 0;
  long long c0 = 0;
  auto process = [&](double lw, float x, bool has_x) {
    const unsigned long long k = double_key(lw);
    if (LEVEL == 0) {
      const double g = (lw - p.log_v0) / p.h;
      a0 += g;
      bool ok;
      if (has_x) ok = x > 0.0f && x < __int_as_float(0x7f800000);
      else ok = fabs(lw) < __longlong_as_double(0x7ff0000000000000LL);
      if (ok) { a1 += g; ++c0; }
    } else if (LEVEL == 1) {
      const double d = (lw - p.log_v0) / p.h - mean;
      a0 += d * d;
    }
    select64_count<LEVEL, GT>(k, pfx, g_hist);
  };
  // four independent loads per thread are in flight before the first is used: with 64 KB of histograms a
  // block the SM holds few warps, so the passes were bound by one memory round trip per element per thread
  constexpr int U = 4;
  const int64_t stride = (int64_t)gridDim.x * G_THREADS * U;
  for (int64_t base = (int64_t)blockIdx.x * G_THREADS * U + threadIdx.x; base < n; base += stride) {
    double lw[U];
    float x[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = base + (int64_t)u * G_THREADS;
      lw[u] = i < n ? __ldcs(v + i) : 0.0;
      x[u] = (LEVEL == 0 && w32 != nullptr && i < n) ? __ldcs(w32 + i) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (base + (int64_t)u * G_THREADS < n) process(lw[u], x[u], w32 != nullptr);
  }
  if (LEVEL == 0) {
    const double s0 = block_sum(a0, red_d), s1 = block_sum(a1, red_d);
    const long long n0 = block_sum(c0, red_i);
    if (threadIdx.x == 0) {
      atomicAdd(&w->sum_g, s0);
      atomicAdd(&w->sum_g_valid, s1);
      atomicAdd((unsigned long long*)&w->cnt_valid, (unsigned long long)n0);
    }
  } else if (LEVEL == 1) {
    const double s0 = block_sum(a0, red_d);
    if (threadIdx.x == 0) atomicAdd(&w->sqdev, s0);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NH * GBINS; i += G_THREADS) {
    const unsigned int c = g_hist[i];
    if (c) atomicAdd((unsigned long long*)(&w->hist[0][0] + i), (unsigned long long)c);
  }
}

// one block per row: walk the level's histograms, extend the prefixes, clear them
__global__ void __launch_bounds__(256)
growth_resolve_kernel(GrowthWS* __restrict__ ws, int level, int64_t n_total, const __grid_constant__ GrowthParams p,
                      double* __restrict__ out, int out_ld) {
  GrowthWS* w = ws + blockIdx.x;
  // warp j resolves target j (eight warps, eight targets, all at once)
  {
    const int j = threadIdx.x >> 5;
    const long long* h = level == 0 ? w->hist[0] : w->hist[j];
    const long long rank = level == 0 ? p.rank[j] : w->rank[j];
    if (select64_resolve(h, level, rank, &w->prefix[j], &w->rank[j]) && level == GLEVELS - 1)
      w->value[j] = (key_double(w->prefix[j]) - p.log_v0) / p.h;
  }
  __threadfence_block();
  __syncthreads();
  // clear the histograms for the next level
  for (int i = threadIdx.x; i < GT * GBINS; i += 256) (&w->hist[0][0])[i] = 0;
  if (threadIdx.x == 0) {
    if (level == 0) w->mean = w->sum_g / (double)n_total;
    if (level == GLEVELS - 1) {
      double* o = out + (int64_t)blockIdx.x * out_ld;
      o[0] = (double)w->cnt_valid;
      o[1] = w->mean;
      o[2] = sqrt(w->sqdev / (double)n_total);
      o[3] = w->cnt_valid > 0 ? w->sum_g_valid / (double)w->cnt_valid : __longlong_as_double(0x7ff8000000000000LL);
      o[4] = w->value[6];
      o[5] = w->value[7];
      for (int q = 0; q < p.n_q; ++q) {
        const double a = w->value[2 * q], b = w->value[2 * q + 1], t = p.frac[q];
        // numpy's _lerp (lib/function_base.py): a + (b-a) t, from the other end for t >= 0.5
        double r = a + (b - a) * t;
        if (t >= 0.5) r = b - (b - a) * (1.0 - t);
        if (t == 0.0 || a == b) r = a;
        o[6 + q] = r;
      }
    }
  }
}

template <int LEVEL>
static void launch_growth_pass(dim3 grid, const double* lw, const float* dT, int64_t n, int64_t ld, int64_t ld_T,
                               GrowthWS* ws, const GrowthParams& p, cudaStream_t st) {
  const size_t smem = (size_t)(LEVEL == 0 ? 1 : GT) * GBINS * sizeof(unsigned int);
  if (smem > 48 * 1024) {
    static bool done[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !done[dev]) {
      cudaFuncSetAttribute(growth_pass_kernel<LEVEL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      done[dev] = true;
    }
  }
  growth_pass_kernel<LEVEL><<<grid, G_THREADS, smem, st>>>(lw, dT, n, ld, ld_T, ws, p);
}

}  // namespace b200

using namespace b200;

extern "C" int64_t b200_growth_workspace_bytes(int64_t rows) {
  return rows < 0 ? 0 : rows * (int64_t)sizeof(GrowthWS);
}

extern "C" int b200_growth_exchange(int32_t phase, int64_t out[5]) {
  B200_REQUIRE(out != nullptr, "growth_exchange: NULL output");
  int64_t io = 0, ic = 0, d_o = 0, dc = 0;
  if (phase == 0) { io = GW_OFF_CNT; ic = 8 + GBINS; d_o = 0; dc = 2; }           // cnt_valid .. hist[0]
  else if (phase >= 1 && phase < GLEVELS) { io = GW_OFF_HIST; ic = (int64_t)GT * GBINS; if (phase == 1) { d_o = 2; dc = 1; } }
  out[0] = io; out[1] = ic; out[2] = d_o; out[3] = dc; out[4] = GW_ROW_WORDS;
  return 0;
}

// phase p in 0..5: (resolve level p-1) + pass p; phase 6: resolve level 5 and write `out`; -1: all.
extern "C" int b200_growth_summary(const double* log_w, const float* data_T, int64_t rows, int64_t n, int64_t ld,
                                   int64_t ld_T, int64_t n_total, double log_v0, int32_t horizon,
                                   const double* quantiles_host, int32_t n_q, void* workspace, double* out,
                                   int32_t phase, void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(rows >= 0 && n >= 0, "growth_summary: negative size");
  if (rows == 0) return 0;
  B200_REQUIRE(log_w != nullptr || n == 0, "growth_summary: log_w is NULL");
  B200_REQUIRE(workspace != nullptr && out != nullptr, "growth_summary: workspace/out is NULL");
  B200_REQUIRE(n_total >= 1 && n <= n_total, "growth_summary: need 1 <= n <= n_total");
  B200_REQUIRE(ld >= n && (data_T == nullptr || ld_T >= n), "growth_summary: ld < n");
  B200_REQUIRE(horizon >= 1, "growth_summary: horizon < 1");
  B200_REQUIRE(n_q >= 0 && n_q <= 3, "growth_summary: 0..3 quantiles per call (got %d)", n_q);
  B200_REQUIRE(n_q == 0 || quantiles_host != nullptr, "growth_summary: quantiles_host is NULL");
  B200_REQUIRE(phase >= -1 && phase <= GLEVELS, "growth_summary: phase out of range");
  if (rows > 65535) return set_error(B200_ELIMIT, "growth_summary: rows=%lld > 65535 per call", (long long)rows);
  GrowthParams p;
  p.log_v0 = log_v0;
  p.h = (double)horizon;
  p.n_q = n_q;
  for (int j = 0; j < GT; ++j) p.rank[j] = 0;
  for (int q = 0; q < 3; ++q) p.frac[q] = 0.0;
  for (int q = 0; q < n_q; ++q) {
    const double qq = quantiles_host[q];
    B200_REQUIRE(qq >= 0.0 && qq <= 1.0, "growth_summary: quantile %g outside [0,1]", qq);
    // Hyndman-Fan type 8 (numpy method="median_unbiased"): alpha = beta = 1/3
    double v = (double)n_total * qq + (1.0 + qq) / 3.0 - 1.0;
    if (v < 0.0) v = 0.0;
    if (v > (double)(n_total - 1)) v = (double)(n_total - 1);
    const long long lo = (long long)floor(v);
    p.rank[2 * q] = lo;
    p.rank[2 * q + 1] = lo + 1 < n_total ? lo + 1 : n_total - 1;
    p.frac[q] = v - (double)lo;
  }
  p.rank[6] = 0;
  p.rank[7] = n_total - 1;

  cudaStream_t st = (cudaStream_t)stream;
  GrowthWS* ws = (GrowthWS*)workspace;
  int64_t want = ((int64_t)sm_count() * 8 + rows - 1) / rows;
  int64_t max_slices = (n + G_THREADS * 8 - 1) / (G_THREADS * 8);
  int64_t slices = want < max_slices ? want : max_slices;
  if (slices < 1) slices = 1;
  dim3 grid((unsigned)slices, (unsigned)rows);
  const int first = phase < 0 ? 0 : phase, last = phase < 0 ? GLEVELS : phase;
  for (int ph = first; ph <= last; ++ph) {
    if (ph == 0) B200_CUDA(cudaMemsetAsync(ws, 0, (size_t)rows * sizeof(GrowthWS), st));
    else growth_resolve_kernel<<<(unsigned)rows, 256, 0, st>>>(ws, ph - 1, n_total, p, out, 6 + n_q);
    if (ph < GLEVELS && n > 0) {
      switch (ph) {
        case 0: launch_growth_pass<0>(grid, log_w, data_T, n, ld, ld_T, ws, p, st); break;
        case 1: launch_growth_pass<1>(grid, log_w, data_T, n, ld, ld_T, ws, p, st); break;
        case 2: launch_growth_pass<2>(grid, log_w, data_T, n, ld, ld_T, ws, p, st); break;
        case 3: launch_growth_pass<3>(grid, log_w, data_T, n, ld, ld_T, ws, p, st); break;
        case 4: launch_growth_pass<4>(grid, log_w, data_T, n, ld, ld_T, ws, p, st); break;
        case 5: launch_growth_pass<5>(grid, log_w, data_T, n, ld, ld_T, ws, p, st); break;
      }
    }
  }
  B200_CUDA(cudaGetLastError());
  return 0;
}
