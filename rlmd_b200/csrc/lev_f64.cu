// Exact fp64 leverage chain: the *_smart_lev / *_fixed_final_lev wealth of the reference
// run under torch.set_default_dtype(float64) (lev/lev_exp.py:160-212, :1042-1093):
//     value = value_0 * m[:, 0];  value = value * m[:, t]          (sequential, fp64)
// discrete: m = table[g][code], the table computed on the host in double;
// GBM:      m = exp(l * x), x fp64, one rounding for the product and the library exp.
// The library is compiled with -fmad=false, so the discrete chain is bit-identical to
// NumPy's sequential fp64 product.
//
// One thread per investor and f64_pt(K) grid points (blockIdx.y walks the tiles of points,
// so registers do not grow with the grid); the thread reads its own outcome row in
// 16-byte pieces.  The wealth after every step goes to dump [G, t_end - t_begin, N]
// (coalesced over investors), or only the state advances.
#include "common.cuh"

namespace b200 {

// grid points per thread: at 8 the GBM kernel (exp's slow path) spills, at 4 it does not
__host__ __device__ constexpr int f64_pt(int K) { return K == 0 ? 4 : 8; }

struct F64Table {
  double m[B200_MAX_GRID][B200_MAX_OUTCOMES];   // discrete: factor of code k; GBM: m[g][0] = l
};

template <int K>   // K = 0: GBM
__global__ void __launch_bounds__(128)
lev_chunk_f64_kernel(const void* __restrict__ outcomes, int64_t ld, const __grid_constant__ F64Table tab, int32_t G,
                     int64_t N, int32_t t_begin, int32_t t_end, double* __restrict__ state, double* __restrict__ dump) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  constexpr int F64_PT = f64_pt(K), KF = K == 0 ? 1 : K;
  const int p0 = blockIdx.y * F64_PT;
  double V[F64_PT], f[F64_PT][KF];
#pragma unroll
  for (int q = 0; q < F64_PT; ++q) {
    const int p = min(p0 + q, G - 1);
    V[q] = state[(int64_t)p * N + i];
#pragma unroll
    for (int k = 0; k < KF; ++k) f[q][k] = tab.m[p][k];
  }
  const int64_t tc = t_end - t_begin;
  auto step = [&](unsigned code, double x, int t) {
#pragma unroll
    for (int q = 0; q < F64_PT; ++q) {
      double m = f[q][0];
      if (K == 0) {
        m = exp(m * x);
      } else {
#pragma unroll
        for (int k = 1; k < KF; ++k) m = code == (unsigned)k ? f[q][k] : m;
      }
      V[q] = V[q] * m;
      if (dump != nullptr && p0 + q < G) __stcs(dump + ((int64_t)(p0 + q) * tc + (t - t_begin)) * N + i, V[q]);
    }
  };
  int t = t_begin;
  if (K == 0) {
    const double* __restrict__ row = (const double*)outcomes + i * ld;
    while (t < t_end) {
      if (((uintptr_t)(row + t) & 15) == 0 && t + 2 <= t_end) {
        const double2 x2 = __ldg(reinterpret_cast<const double2*>(row + t));
        step(0, x2.x, t);
        step(0, x2.y, t + 1);
        t += 2;
      } else {
        step(0, __ldg(row + t), t);
        ++t;
      }
    }
  } else {
    const uint8_t* __restrict__ row = (const uint8_t*)outcomes + i * ld;
    while (t < t_end) {
      if (((uintptr_t)(row + t) & 15) == 0 && t + 16 <= t_end) {      // 16 outcomes per load
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(row + t));
        const unsigned words[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int b = 0; b < 16; ++b) step((words[b >> 2] >> (8 * (b & 3))) & 0xffu, 0.0, t + b);
        t += 16;
      } else {
        step(__ldg(row + t), 0.0, t);
        ++t;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < F64_PT; ++q)
    if (p0 + q < G) state[(int64_t)(p0 + q) * N + i] = V[q];
}

}  // namespace b200

using namespace b200;

extern "C" int b200_lev_chunk_f64(const b200_lev_desc* desc, const void* outcomes, const double* factors_host,
                                  int32_t t_begin, int32_t t_end, double* state, double* dump, void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(desc != nullptr, "lev_chunk_f64: desc is NULL");
  const b200_lev_desc& d = *desc;
  B200_REQUIRE(d.kind == B200_LEV_DISCRETE || d.kind == B200_LEV_GBM, "lev_chunk_f64: unknown kind %d", d.kind);
  B200_REQUIRE(d.source == B200_SRC_STREAM, "lev_chunk_f64: outcomes are streamed (no Philox source)");
  B200_REQUIRE(d.n_investors >= 0 && d.horizon >= 1, "lev_chunk_f64: need n_investors >= 0 and horizon >= 1");
  B200_REQUIRE(d.n_grid >= 1 && d.n_grid <= B200_MAX_GRID, "lev_chunk_f64: n_grid must be in 1..%d", B200_MAX_GRID);
  B200_REQUIRE(d.kind == B200_LEV_GBM || (d.n_outcomes >= 2 && d.n_outcomes <= B200_MAX_OUTCOMES),
               "lev_chunk_f64: n_outcomes must be in 2..%d", B200_MAX_OUTCOMES);
  B200_REQUIRE(d.outcome_bits == 0 || d.outcome_bits == 8, "lev_chunk_f64: outcomes are uint8 codes or fp64 x");
  B200_REQUIRE(d.ld_outcomes >= d.horizon, "lev_chunk_f64: ld_outcomes < horizon");
  B200_REQUIRE(0 <= t_begin && t_begin < t_end && t_end <= d.horizon,
               "lev_chunk_f64: need 0 <= t_begin < t_end <= horizon");
  B200_REQUIRE(factors_host != nullptr, "lev_chunk_f64: factors is NULL");
  if (d.n_investors == 0) return 0;
  B200_REQUIRE(outcomes != nullptr && state != nullptr, "lev_chunk_f64: outcomes/state is NULL");
  const int K = d.kind == B200_LEV_GBM ? 1 : d.n_outcomes;
  F64Table tab;
  for (int g = 0; g < B200_MAX_GRID; ++g)
    for (int k = 0; k < B200_MAX_OUTCOMES; ++k) tab.m[g][k] = g < d.n_grid && k < K ? factors_host[g * K + k] : 0.0;
  const int pt = f64_pt(d.kind == B200_LEV_GBM ? 0 : K);
  const dim3 grid((unsigned)((d.n_investors + 127) / 128), (unsigned)((d.n_grid + pt - 1) / pt));
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t N = d.n_investors, ld = d.ld_outcomes;
  if (d.kind == B200_LEV_GBM)
    lev_chunk_f64_kernel<0><<<grid, 128, 0, st>>>(outcomes, ld, tab, d.n_grid, N, t_begin, t_end, state, dump);
  else if (K == 2)
    lev_chunk_f64_kernel<2><<<grid, 128, 0, st>>>(outcomes, ld, tab, d.n_grid, N, t_begin, t_end, state, dump);
  else if (K == 3)
    lev_chunk_f64_kernel<3><<<grid, 128, 0, st>>>(outcomes, ld, tab, d.n_grid, N, t_begin, t_end, state, dump);
  else
    lev_chunk_f64_kernel<4><<<grid, 128, 0, st>>>(outcomes, ld, tab, d.n_grid, N, t_begin, t_end, state, dump);
  return check_cuda(cudaGetLastError(), "lev_chunk_f64 launch");
}
