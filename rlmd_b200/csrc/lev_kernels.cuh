// Device code shared by the leverage-sweep translation units.
//
// Reference: lev/lev_exp.py - the per-leverage loop of *_fixed_final_lev
// (:83-87, :539-545, :963-967, :1158-1168) and the sequential chain of
// *_smart_lev (:167-175, :629-640, :1048-1055, :1258-1273).
//
// CHAIN (discrete): one thread per investor, G wealth registers, the exact fp32
//   product ((V0*m_0)*m_1)*... in time order.  Outcome bytes [N,ld] are staged
//   through shared memory in [128 investors x 128 steps] tiles by TMA
//   (cp.async.bulk.tensor.2d, 128-byte swizzle => the per-thread row reads are
//   16-byte LDS without bank conflicts) behind a ring of mbarriers.  Rows whose
//   stride or base is not 16-byte aligned take a cooperative plain-load path
//   into the same swizzled layout.  The same kernel serves the per-step series
//   (*_smart_lev): it can start from a saved state, stop at any step, and dump
//   the wealth after every step into a [G, steps, N] chunk buffer.
#pragma once
#include <cuda.h>

#include <cmath>
#include <cstring>

#include "common.cuh"

namespace b200 {

constexpr int TILE_ROWS = 128;   // investors per block
constexpr int TILE_BYTES = 128;  // bytes of one investor's row per tile (swizzle span)
constexpr int STAGES = 4;
constexpr int TILE_SMEM = TILE_ROWS * TILE_BYTES;  // 16 KB

struct FactorTable {
  float m[B200_MAX_OUTCOMES][32];  // [k][g] for one grid tile of <= 32 points
};
struct Thresholds {
  uint32_t t[B200_MAX_OUTCOMES];
};

// ------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// 16-byte chunk `c` of tile row `r` under the 128-byte swizzle.
__device__ __forceinline__ uint32_t swz(int r, int c) { return (uint32_t)(r * TILE_BYTES + ((c ^ (r & 7)) << 4)); }

// ------------------------------------------------------- one chain step
// Two bit-identical ways to apply w[g] *= m[code][g] for the whole grid tile
// (one IEEE fp32 multiply per path-step; they differ in how the factor is
// selected, i.e. in which pipes they load - DESIGN.md "chain variants"):
//   V_FSEL : per g, (K-1) FSEL from constant-bank factors + 1 FMUL
//   V_LDS  : factor rows m[code][*] fetched from a shared-memory table with
//            LDS.128 (lanes that saw the same code share the fetch) + FMUL2
//   V_FMA  : (K <= 3) the code byte, moved to the top byte of a word, IS the
//            float c in {0, 2^-125 (code 1), 2^-123 (code 2)}; the factor of the
//            highest code is produced on the FMA pipe as fma(c, A_g, m[0][g])
//            with A_g (row 3 of the table) chosen on the host so that the single
//            rounding lands exactly on m[K-1][g] (fma_deltas() verifies every
//            entry bit for bit, else the launch falls back).  K = 3 patches
//            code 1 in with one FSEL; K = 2 splits the grid tile between FSEL
//            and FMA selection so that the ALU and FMA pipes fill together.
//            FFMA2/FMUL2 halve the issue slots.
enum { V_FSEL = 0, V_LDS = 1, V_FMA = 2 };

// Selector word of one step: the code itself, or code << 24 for V_FMA.
template <int V>
__device__ __forceinline__ uint32_t sel_from_word(uint32_t wd, int b) {
  return V == V_FMA ? __byte_perm(wd, 0u, (uint32_t)((b << 12) | 0x444)) : ((wd >> (8 * b)) & 0xffu);
}
template <int V>
__device__ __forceinline__ uint32_t sel_from_code(uint32_t code) { return V == V_FMA ? code << 24 : code; }

// K = 2: grid points [0, fma_nsel) are selected by FSEL, the rest by FFMA.
__host__ __device__ constexpr int fma_nsel(int GT) { return ((GT * 11 / 20) + 1) & ~1; }

template <int GT>
struct GridTile {
  static constexpr int PAD = (GT + 3) & ~3;                       // floats per table row, multiple of 4
  static constexpr int STRIDE = (PAD % 16 == 0) ? PAD + 4 : PAD;  // rows of different codes on disjoint banks
};

template <int GT, int K, int V>
__device__ __forceinline__ void chain_step(float (&w)[GT], const FactorTable& f, const float* __restrict__ tab,
                                           uint32_t code) {
  if (V == V_LDS) {
    constexpr int S = GridTile<GT>::STRIDE;
    const float4* __restrict__ row = reinterpret_cast<const float4*>(tab + code * S);
#pragma unroll
    for (int c = 0; c < GridTile<GT>::PAD / 4; ++c) {
      const float4 m = row[c];
      const int g = 4 * c;
      if (g + 1 < GT) {
        const float2 r = __fmul2_rn(make_float2(w[g], w[g + 1]), make_float2(m.x, m.y));
        w[g] = r.x; w[g + 1] = r.y;
      } else if (g < GT) {
        w[g] = __fmul_rn(w[g], m.x);
      }
      if (g + 3 < GT) {
        const float2 r = __fmul2_rn(make_float2(w[g + 2], w[g + 3]), make_float2(m.z, m.w));
        w[g + 2] = r.x; w[g + 3] = r.y;
      } else if (g + 2 < GT) {
        w[g + 2] = __fmul_rn(w[g + 2], m.z);
      }
    }
  } else if (V == V_FMA) {
    const float c = __uint_as_float(code);  // code << 24 read as a float
    const bool hit = (K == 2) ? (code != 0u) : (code == 0x01000000u);
    constexpr int NSEL = (K == 2) ? fma_nsel(GT) : 0;
    float m[GT];
#pragma unroll
    for (int g = 0; g < GT; g += 2) {
      if (g + 1 < GT) {
        if (g >= NSEL) {
          const float2 r = __ffma2_rn(make_float2(c, c), make_float2(f.m[3][g], f.m[3][g + 1]),
                                      make_float2(f.m[0][g], f.m[0][g + 1]));
          m[g] = r.x; m[g + 1] = r.y;
        }
        if (K == 3 || g < NSEL) {
          m[g] = hit ? f.m[1][g] : (K == 2 ? f.m[0][g] : m[g]);
          m[g + 1] = hit ? f.m[1][g + 1] : (K == 2 ? f.m[0][g + 1] : m[g + 1]);
        }
        const float2 r = __fmul2_rn(make_float2(w[g], w[g + 1]), make_float2(m[g], m[g + 1]));
        w[g] = r.x; w[g + 1] = r.y;
      } else {
        float mm = __fmaf_rn(c, f.m[3][g], f.m[0][g]);
        if (K == 3) mm = hit ? f.m[1][g] : mm;
        w[g] = __fmul_rn(w[g], mm);
      }
    }
  } else {
    const bool is1 = code == 1, is2 = code == 2, is3 = code == 3;
#pragma unroll
    for (int g = 0; g < GT; ++g) {
      float m = f.m[0][g];
      m = (K == 2 ? code != 0 : is1) ? f.m[1][g] : m;
      if (K >= 3) m = is2 ? f.m[2][g] : m;
      if (K >= 4) m = is3 ? f.m[3][g] : m;
      w[g] = __fmul_rn(w[g], m);
    }
  }
}

template <int GT, int K>
__device__ __forceinline__ void fill_table(float* tab, const FactorTable& f) {
  constexpr int S = GridTile<GT>::STRIDE;
  for (int i = threadIdx.x; i < K * S; i += blockDim.x) {
    const int k = i / S, g = i - k * S;
    tab[i] = g < GT ? f.m[k][g] : 1.0f;
  }
}

// Arguments common to the chain kernels.  Steps [t_begin, t_end) are applied to
// the state (V0 when state_in is NULL); the wealth after step t goes to
// dump[(g * (t_end - t_begin) + (t - t_begin)) * ldT + investor] when DUMP.
struct ChainParams {
  int32_t t_begin, t_end;
  int32_t G;       // live grid points of this tile (<= GT)
  float V0;
  int64_t N;
  int64_t ldT;     // row stride of state / dump
  const float* state_in;
  float* state_out;
  float* dump;
};

template <int GT, bool DUMP>
__device__ __forceinline__ void dump_step(const float (&w)[GT], const ChainParams& p, int t, int64_t row) {
  if (DUMP) {
    const int64_t tc = p.t_end - p.t_begin;
#pragma unroll
    for (int g = 0; g < GT; ++g)
      if (g < p.G) __stcs(p.dump + ((int64_t)g * tc + (t - p.t_begin)) * p.ldT + row, w[g]);
  }
}

// --------------------------------------------- CHAIN, discrete, streamed
// USE_TMA: tiles arrive by cp.async.bulk.tensor; otherwise all threads copy.
template <int GT, int K, int V, bool USE_TMA, bool DUMP>
__global__ void __launch_bounds__(TILE_ROWS)
chain_discrete_stream_kernel(const __grid_constant__ CUtensorMap tmap, const uint8_t* __restrict__ outcomes,
                             int64_t ld, const __grid_constant__ FactorTable f,
                             const __grid_constant__ ChainParams p, const int stages) {
  extern __shared__ __align__(1024) uint8_t tiles[];
  __shared__ __align__(8) uint64_t full[STAGES];
  __shared__ __align__(16) float tab[V == V_LDS ? K * GridTile<GT>::STRIDE : 4];

  const int tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * TILE_ROWS;
  const int64_t row = row0 + tid;
  const bool live = row < p.N;
  const int nsteps = p.t_end - p.t_begin;
  const int ntiles = (nsteps + TILE_BYTES - 1) / TILE_BYTES;

  if (V == V_LDS) fill_table<GT, K>(tab, f);
  if (USE_TMA) {
    if (tid == 0) {
      for (int s = 0; s < stages; ++s) mbar_init(&full[s], 1);
      fence_barrier_init();
    }
    __syncthreads();
    if (tid == 0) {
      const int pre = ntiles < stages ? ntiles : stages;
      for (int s = 0; s < pre; ++s) {
        mbar_expect_tx(&full[s], TILE_SMEM);
        tma_load_2d(tiles + s * TILE_SMEM, &tmap, &full[s], p.t_begin + s * TILE_BYTES, (int)row0);
      }
    }
  } else {
    __syncthreads();
  }

  float w[GT];
#pragma unroll
  for (int g = 0; g < GT; ++g) w[g] = (p.state_in != nullptr && live && g < p.G) ? p.state_in[(int64_t)g * p.ldT + row] : p.V0;

  int s = 0;
  uint32_t phase = 0;
  for (int kt = 0; kt < ntiles; ++kt) {
    uint8_t* tile = tiles + s * TILE_SMEM;
    const int t0 = p.t_begin + kt * TILE_BYTES;
    if (USE_TMA) {
      mbar_wait(&full[s], phase);
    } else {
      // cooperative copy: consecutive threads read consecutive bytes of a row
      __syncthreads();
      for (int idx = tid; idx < TILE_ROWS * TILE_BYTES; idx += TILE_ROWS) {
        const int r = idx >> 7, b = idx & 127;
        const int64_t rr = row0 + r;
        uint8_t v = 0;
        if (rr < p.N && t0 + b < p.t_end) v = outcomes[rr * ld + t0 + b];
        tile[swz(r, b >> 4) + (b & 15)] = v;
      }
      __syncthreads();
    }
    const int steps = min(TILE_BYTES, p.t_end - t0);
    if (steps == TILE_BYTES) {
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        const uint4 q = *reinterpret_cast<const uint4*>(tile + swz(tid, c));
        const uint32_t wd[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            chain_step<GT, K, V>(w, f, tab, sel_from_word<V>(wd[j], b));
            if (DUMP && live) dump_step<GT, DUMP>(w, p, t0 + c * 16 + j * 4 + b, row);
          }
        }
      }
    } else {
#pragma unroll 1
      for (int t = 0; t < steps; ++t) {
        const uint32_t code = tile[swz(tid, t >> 4) + (t & 15)];
        chain_step<GT, K, V>(w, f, tab, sel_from_code<V>(code));
        if (DUMP && live) dump_step<GT, DUMP>(w, p, t0 + t, row);
      }
    }
    if (USE_TMA) {
      __syncthreads();  // every thread is done with stage s
      if (tid == 0 && kt + stages < ntiles) {
        mbar_expect_tx(&full[s], TILE_SMEM);
        tma_load_2d(tile, &tmap, &full[s], p.t_begin + (kt + stages) * TILE_BYTES, (int)row0);
      }
      if (++s == stages) { s = 0; phase ^= 1u; }
    }
  }

  if (live) {
#pragma unroll
    for (int g = 0; g < GT; ++g)
      if (g < p.G) p.state_out[(int64_t)g * p.ldT + row] = w[g];
  }
}

// ------------------------------------------------- Philox outcome draws
// Four consecutive time steps share one Philox block: counter =
// (investor lo, investor hi, t/4, TAG), key = seed.  Code = #{k: u >= thr[k]}.
template <int K>
__device__ __forceinline__ uint32_t draw_code(uint32_t u, const Thresholds& th) {
  uint32_t c = (u >= th.t[0]);
  if (K >= 3) c += (u >= th.t[1]);
  if (K >= 4) c += (u >= th.t[2]);
  return c;
}

// t_begin must be a multiple of 4 (the host enforces it).
template <int GT, int K, int V, bool DUMP>
__global__ void __launch_bounds__(128)
chain_discrete_philox_kernel(const __grid_constant__ FactorTable f, const __grid_constant__ Thresholds th,
                             const __grid_constant__ PhiloxKeys keys, int64_t investor_offset,
                             const __grid_constant__ ChainParams p) {
  __shared__ __align__(16) float tab[V == V_LDS ? K * GridTile<GT>::STRIDE : 4];
  if (V == V_LDS) {
    fill_table<GT, K>(tab, f);
    __syncthreads();
  }
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= p.N) return;
  const uint64_t id = (uint64_t)(row + investor_offset);
  const uint32_t c0 = (uint32_t)id, c1 = (uint32_t)(id >> 32);
  float w[GT];
#pragma unroll
  for (int g = 0; g < GT; ++g) w[g] = (p.state_in != nullptr && g < p.G) ? p.state_in[(int64_t)g * p.ldT + row] : p.V0;
  const int j0 = p.t_begin >> 2, j1 = p.t_end >> 2;
#pragma unroll 2
  for (int j = j0; j < j1; ++j) {
    const Philox4 r = philox4x32_10(c0, c1, (uint32_t)j, PHILOX_TAG_LEV, keys);
    const uint32_t u[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      chain_step<GT, K, V>(w, f, tab, sel_from_code<V>(draw_code<K>(u[b], th)));
      dump_step<GT, DUMP>(w, p, 4 * j + b, row);
    }
  }
  if (p.t_end & 3) {
    const Philox4 r = philox4x32_10(c0, c1, (uint32_t)j1, PHILOX_TAG_LEV, keys);
    const uint32_t u[4] = {r.x, r.y, r.z, r.w};
    for (int b = 0; b < (p.t_end & 3); ++b) {
      chain_step<GT, K, V>(w, f, tab, sel_from_code<V>(draw_code<K>(u[b], th)));
      dump_step<GT, DUMP>(w, p, 4 * j1 + b, row);
    }
  }
#pragma unroll
  for (int g = 0; g < GT; ++g)
    if (g < p.G) p.state_out[(int64_t)g * p.ldT + row] = w[g];
}

// ------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// [n_rows, row_elems] view with 128-byte x 128-row boxes, 128B swizzle.
int make_row_tile_map(CUtensorMap* map, const void* base, int64_t n_rows, int64_t row_elems, int64_t ld_elems,
                      int elem_bytes);

inline bool tma_ok(const void* base, int64_t ld_bytes, int64_t n_rows) {
  return ((uintptr_t)base % 16 == 0) && (ld_bytes % 16 == 0) && n_rows < ((int64_t)1 << 31);
}

// TMA ring depth of the chain kernels (1..STAGES); B200_CHAIN_STAGES overrides for tuning.
int chain_stages();

// One grid tile (<= 32 points) of a discrete CHAIN sweep; defined per K in
// lev_chain_k{2,3,4}.cu so that the instantiations compile in parallel.
struct ChainLaunch {
  const b200_lev_desc* d;
  const uint8_t* outcomes;
  FactorTable f;
  ChainParams p;
  int variant;  // 1 = V_FSEL, 2 = V_LDS, 3 = V_FMA (0 = default for this K)
  cudaStream_t st;
};
template <int K>
int chain_discrete_launch(const ChainLaunch& a);

// ---- generic launcher body (included by the per-K translation units) ----
template <int GT, int K, int V, bool DUMP>
static int chain_launch_impl(const ChainLaunch& a) {
  const b200_lev_desc& d = *a.d;
  const int64_t N = d.n_investors;
  if (d.source == B200_SRC_PHILOX) {
    Thresholds th;
    for (int k = 0; k < B200_MAX_OUTCOMES; ++k) th.t[k] = d.thresholds[k];
    const unsigned blocks = (unsigned)((N + 127) / 128);
    chain_discrete_philox_kernel<GT, K, V, DUMP><<<blocks, 128, 0, a.st>>>(a.f, th, philox_keys(d.seed), d.investor_offset, a.p);
    return check_cuda(cudaGetLastError(), "chain_discrete_philox launch");
  }
  const unsigned blocks = (unsigned)((N + TILE_ROWS - 1) / TILE_ROWS);
  CUtensorMap map;
  memset(&map, 0, sizeof(map));
  if (tma_ok(a.outcomes, d.ld_outcomes, N)) {
    int rc = make_row_tile_map(&map, a.outcomes, N, d.horizon, d.ld_outcomes, 1);
    if (rc) return rc;
    // The chain is issue-bound, not HBM-bound: a short ring leaves room for more
    // resident blocks per SM (the warps hide the ALU latency of the dependent chain).
    const int stages = chain_stages();
    auto kern = chain_discrete_stream_kernel<GT, K, V, true, DUMP>;
    B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, STAGES * TILE_SMEM));
    kern<<<blocks, TILE_ROWS, stages * TILE_SMEM, a.st>>>(map, a.outcomes, d.ld_outcomes, a.f, a.p, stages);
  } else {
    chain_discrete_stream_kernel<GT, K, V_FSEL, false, DUMP><<<blocks, TILE_ROWS, TILE_SMEM, a.st>>>(
        map, a.outcomes, d.ld_outcomes, a.f, a.p, 1);
  }
  return check_cuda(cudaGetLastError(), "chain_discrete_stream launch");
}

template <int K, int V, bool DUMP>
static int chain_launch_gt(const ChainLaunch& a) {
  const int g = a.p.G;
  if (g <= 4) return chain_launch_impl<4, K, V, DUMP>(a);
  if (g <= 10) return chain_launch_impl<10, K, V, DUMP>(a);
  if (g <= 20) return chain_launch_impl<20, K, V, DUMP>(a);
  return chain_launch_impl<32, K, V, DUMP>(a);
}

// Default variant, from the B200 measurements in profiles/r01_kernels_*.jsonl
// (investor-steps/s at G = 10, 1e6 x 1e4):  streamed dice FSEL 7.7e11, LDS 9.0e11,
// FMA 1.28e12; streamed coin FSEL 1.58e12, LDS 9.0e11, FMA 1.68e12; Philox dice
// FSEL 5.6e11, LDS 8.9e11, FMA 6.7e11 (the generator already loads the FMA and ALU
// pipes, so the shared-memory table wins there).
// Fills row 3 of the table with the scaled FMA deltas of V_FMA; false when some
// entry cannot be reproduced bit for bit by one fused multiply-add.
inline bool fma_deltas(FactorTable& f, int K, int g_cnt) {
  if (K > 3) return false;
  const int scale_exp = (K == 2) ? 125 : 123;              // 1 / c of the highest code
  const float c = ldexpf(1.0f, -scale_exp);
  for (int g = 0; g < 32; ++g) {
    f.m[3][g] = 0.0f;
    if (g >= g_cnt) continue;
    const float f0 = f.m[0][g], ft = f.m[K - 1][g];
    uint32_t want, got;
    memcpy(&want, &ft, 4);
    const float a0 = (float)((double)ft - (double)f0);
    const float cand[3] = {a0, nextafterf(a0, INFINITY), nextafterf(a0, -INFINITY)};
    bool ok = false;
    for (int i = 0; i < 3 && !ok; ++i) {
      const float as = ldexpf(cand[i], scale_exp);
      if (!std::isfinite(as)) continue;
      const float r1 = fmaf(c, as, f0), r0 = fmaf(0.0f, as, f0);
      memcpy(&got, &r1, 4);
      uint32_t b0, w0;
      memcpy(&b0, &r0, 4);
      memcpy(&w0, &f0, 4);
      if (got == want && b0 == w0) { f.m[3][g] = as; ok = true; }
    }
    if (!ok) return false;
  }
  return true;
}

template <int K>
static int chain_launch_all(const ChainLaunch& a0) {
  ChainLaunch a = a0;
  int v = a.variant;
  const int fallback = (K == 2) ? 1 : 2;
  if (v == 0) v = (K <= 3 && a.d->source != B200_SRC_PHILOX) ? 3 : fallback;
  if (v == 3 && !fma_deltas(a.f, K, a.p.G)) v = fallback;
  const bool dump = a.p.dump != nullptr;
  if constexpr (K <= 3) {
    if (v == 3) return dump ? chain_launch_gt<K, V_FMA, true>(a) : chain_launch_gt<K, V_FMA, false>(a);
  }
  if (v == 2) return dump ? chain_launch_gt<K, V_LDS, true>(a) : chain_launch_gt<K, V_LDS, false>(a);
  return dump ? chain_launch_gt<K, V_FSEL, true>(a) : chain_launch_gt<K, V_FSEL, false>(a);
}

// GBM: the running sum S of the log-returns, 32 steps in fp32 relative to the fp64 base, then
// folded into the base.  The LOG sweep, the series chunks (lev_sweep.cu) and the sum route
// (gbm_sum.cu) all accumulate through this one struct, so their S agree bit for bit.
struct GbmAcc {
  double S = 0.0, Smax = 0.0, Smin = 0.0;  // running sum and its extremes (t >= 0; start value 0)
  float p = 0.f, pmax = -3.0e38f, pmin = 3.0e38f;
  __device__ __forceinline__ void step(float x) {
    p += x;
    pmax = fmaxf(pmax, p);
    pmin = fminf(pmin, p);
  }
  // two steps: the running extremes take both partial sums in ONE three-input min / max each
  // (FMNMX3, sm_100) - 4 instructions per pair instead of 6, the same values bit for bit
  __device__ __forceinline__ void step2(float x0, float x1) {
    const float p1 = p + x0;
    p = p1 + x1;
    asm("max.f32 %0, %0, %1, %2;" : "+f"(pmax) : "f"(p1), "f"(p));
    asm("min.f32 %0, %0, %1, %2;" : "+f"(pmin) : "f"(p1), "f"(p));
  }
  __device__ __forceinline__ void fold() {
    Smax = fmax(Smax, S + (double)pmax);
    Smin = fmin(Smin, S + (double)pmin);
    S += (double)p;
    p = 0.f; pmax = -3.0e38f; pmin = 3.0e38f;
  }
};

}  // namespace b200
