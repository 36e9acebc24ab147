// Per-step series of the three-outcome gamble (the dice, with or without insurance) from the
// count-tuple lattice (dice_smart_lev(..., method="tuples"); DESIGN.md section 6.11).
//
// After step t an investor with a up-moves, b down-moves and c = t+1-a-b mid-moves holds
// V0 u^a d^b m^c at EVERY leverage, so the 12 statistics of every leverage at step t follow
// from one integer histogram over the (a, b) cells occupied at t:
//   bounds : one read of the codes -> amin/amax/bmin/bmax of every step (and each investor's
//            running (a, b)); the host lays the steps' boxes out flat and plans chunks from them;
//   count  : a second read -> each step's box [amax-amin+1][bmax-bmin+1], one global
//            reduction per investor-step;
//   stats  : per (step, leverage) a block selects the ranks on the log wealth
//            x = log V0 + a log u + b log d + c log m (fl32(exp(x)) is monotone in x, so the
//            r-th smallest wealth is fl32(exp(r-th smallest x))), then fp64 moments.
// Wealth is not monotone in one count, so the ranks come from a weighted select on x: a
// histogram of x over the occupied cells' [xmin, xmax], refined inside the bin that holds the
// rank until that bin holds few enough cells to rank them one against another.  The bin of x
// is clamp(floor((x - lo) * scale)), monotone in x, so a bin holds exactly a run of ranks.
#include <cfloat>
#include <climits>
#include <cmath>

#include "common.cuh"

namespace b200 {

constexpr int DL_THREADS = 256;
constexpr int DL_TT = 32;        // steps per tile: two 16-byte loads of a row

// (up, down) bit masks of the tile `tile` of one row: bit s = step 32 * tile + s, for the steps in [t_lo, t_hi)
// (code 0 = up, 1 = down, anything else = mid; other bits are whatever the row holds there and are never read)
__device__ __forceinline__ void dice_tile_masks(const uint8_t* __restrict__ row, int tile, int t_lo, int t_hi,
                                                bool aligned, uint32_t& up, uint32_t& dn) {
  const int t0 = tile * DL_TT;
  up = 0u;
  dn = 0u;
  if (aligned) {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      if (t0 + 16 * q >= t_hi) break;      // (ld is a multiple of 16 >= horizon: a started piece is in the row)
      const uint4 w4 = __ldg(reinterpret_cast<const uint4*>(row + t0 + 16 * q));
      const uint32_t w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const int s = 16 * q + k;
        const uint32_t code = (w[k >> 2] >> (8 * (k & 3))) & 0xffu;
        up |= (uint32_t)(code == 0u) << s;
        dn |= (uint32_t)(code == 1u) << s;
      }
    }
  } else {
    for (int t = t_lo; t < t_hi; ++t) {
      const uint32_t code = __ldg(row + t);
      up |= (uint32_t)(code == 0u) << (t - t0);
      dn |= (uint32_t)(code == 1u) << (t - t0);
    }
  }
}

// bounds rows: 0 amin, 1 amax, 2 bmin, 3 bmax; column i = step t_begin + i
template <int R>
__global__ void __launch_bounds__(DL_THREADS)
dice_bounds_kernel(const uint8_t* __restrict__ outcomes, int64_t N, int64_t ld, bool aligned, int32_t t_begin,
                   int32_t t_end, int32_t* __restrict__ ab_state, int32_t* __restrict__ bounds, int64_t ld_bounds) {
  __shared__ int32_t sh[4][DL_TT];
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t i0 = (int64_t)blockIdx.x * DL_THREADS * R + tid;
  int a[R], b[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t i = i0 + (int64_t)r * DL_THREADS;
    a[r] = (i < N && t_begin > 0) ? ab_state[i] : 0;
    b[r] = (i < N && t_begin > 0) ? ab_state[N + i] : 0;
  }
  for (int tile = t_begin / DL_TT; tile * DL_TT < t_end; ++tile) {
    const int t0 = tile * DL_TT;
    const int t_lo = max(t_begin, t0), t_hi = min(t_end, t0 + DL_TT);
    if (tid < 4 * DL_TT) sh[tid / DL_TT][tid % DL_TT] = (tid / DL_TT) % 2 == 0 ? INT_MAX : -1;
    __syncthreads();
    uint32_t up[R], dn[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int64_t i = i0 + (int64_t)r * DL_THREADS;
      up[r] = dn[r] = 0u;
      if (i < N) dice_tile_masks(outcomes + i * ld, tile, t_lo, t_hi, aligned, up[r], dn[r]);
    }
    for (int t = t_lo; t < t_hi; ++t) {
      const int s = t - t0;
      int alo = INT_MAX, ahi = -1, blo = INT_MAX, bhi = -1;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (i0 + (int64_t)r * DL_THREADS >= N) continue;
        a[r] += (int)((up[r] >> s) & 1u);
        b[r] += (int)((dn[r] >> s) & 1u);
        alo = min(alo, a[r]); ahi = max(ahi, a[r]); blo = min(blo, b[r]); bhi = max(bhi, b[r]);
      }
      alo = __reduce_min_sync(0xffffffffu, alo);
      ahi = __reduce_max_sync(0xffffffffu, ahi);
      blo = __reduce_min_sync(0xffffffffu, blo);
      bhi = __reduce_max_sync(0xffffffffu, bhi);
      if (lane == 0 && ahi >= 0) {
        atomicMin(&sh[0][s], alo); atomicMax(&sh[1][s], ahi);
        atomicMin(&sh[2][s], blo); atomicMax(&sh[3][s], bhi);
      }
    }
    __syncthreads();
    if (tid < 4 * DL_TT) {
      const int q = tid / DL_TT, s = tid % DL_TT, t = t0 + s;
      if (t >= t_lo && t < t_hi && sh[q][s] != (q % 2 == 0 ? INT_MAX : -1)) {
        int32_t* dst = bounds + (int64_t)q * ld_bounds + (t - t_begin);
        if (q % 2 == 0) atomicMin(dst, sh[q][s]); else atomicMax(dst, sh[q][s]);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t i = i0 + (int64_t)r * DL_THREADS;
    if (i < N) { ab_state[i] = a[r]; ab_state[N + i] = b[r]; }
  }
}

// cell (a, b) of step t_begin + i is hist[offsets[i] + (a - amin) * (bmax - bmin + 1) + (b - bmin)]
template <int R>
__global__ void __launch_bounds__(DL_THREADS)
dice_count_kernel(const uint8_t* __restrict__ outcomes, int64_t N, int64_t ld, bool aligned, int32_t t_begin,
                  int32_t t_end, int32_t* __restrict__ ab_state, const int32_t* __restrict__ bounds, int64_t ld_bounds,
                  const int64_t* __restrict__ offsets, int32_t* __restrict__ hist) {
  __shared__ int64_t s_base[DL_TT];
  __shared__ int32_t s_wb[DL_TT];
  const int tid = threadIdx.x;
  const int64_t i0 = (int64_t)blockIdx.x * DL_THREADS * R + tid;
  int a[R], b[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t i = i0 + (int64_t)r * DL_THREADS;
    a[r] = (i < N && t_begin > 0) ? ab_state[i] : 0;
    b[r] = (i < N && t_begin > 0) ? ab_state[N + i] : 0;
  }
  for (int tile = t_begin / DL_TT; tile * DL_TT < t_end; ++tile) {
    const int t0 = tile * DL_TT;
    const int t_lo = max(t_begin, t0), t_hi = min(t_end, t0 + DL_TT);
    __syncthreads();       // the previous tile is done with s_base / s_wb
    if (tid < DL_TT && t0 + tid >= t_lo && t0 + tid < t_hi) {
      const int64_t c = t0 + tid - t_begin;
      const int32_t amin = bounds[c], bmin = bounds[2 * ld_bounds + c];
      const int32_t wb = bounds[3 * ld_bounds + c] - bmin + 1;
      s_wb[tid] = wb;
      s_base[tid] = offsets[c] - (int64_t)amin * wb - bmin;
    }
    __syncthreads();
    uint32_t up[R], dn[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int64_t i = i0 + (int64_t)r * DL_THREADS;
      up[r] = dn[r] = 0u;
      if (i < N) dice_tile_masks(outcomes + i * ld, tile, t_lo, t_hi, aligned, up[r], dn[r]);
    }
    for (int t = t_lo; t < t_hi; ++t) {
      const int s = t - t0;
      const int64_t base = s_base[s];
      const int wb = s_wb[s];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (i0 + (int64_t)r * DL_THREADS >= N) continue;
        a[r] += (int)((up[r] >> s) & 1u);
        b[r] += (int)((dn[r] >> s) & 1u);
        atomicAdd(hist + (base + (int64_t)a[r] * wb + b[r]), 1);
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t i = i0 + (int64_t)r * DL_THREADS;
    if (i < N) { ab_state[i] = a[r]; ab_state[N + i] = b[r]; }
  }
}

constexpr int SEL_BINS = 1024;   // bins of x per select level
constexpr int SEL_CAP = 512;     // cells of a target's bin ranked one against another
constexpr int SEL_LEVELS = 4;    // histogram levels before the step's select gives up (the leverage keeps the chain)
enum { SEL_ACTIVE = 0, SEL_GATHER = 1, SEL_DONE = 2, SEL_FAIL = 3 };

struct DiceLogs {
  double lu[B200_MAX_GRID], ld[B200_MAX_GRID], lm[B200_MAX_GRID];    // log u, log d, log m per leverage
};

// log V0 + a log u + b log d + c log m in fp64, left to right (the library is built with -fmad=false)
__device__ __forceinline__ double dice_x(double lv0, double lu, double ld, double lm, int t, int a, int b) {
  return lv0 + (double)a * lu + (double)b * ld + (double)(t + 1 - a - b) * lm;
}
__device__ __forceinline__ double dice_value(double x) { return (double)__double2float_rn(exp(x)); }

__device__ __forceinline__ int sel_bin(double x, double lo, double scale) {
  const double y = fmin(fmax(floor((x - lo) * scale), 0.0), (double)(SEL_BINS - 1));
  return (int)y;
}

template <typename T>
__device__ __forceinline__ T block_reduce(T v, T* scratch, int op) {    // op 0: sum, 1: min, 2: max (fixed order)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const T u = __shfl_xor_sync(0xffffffffu, v, o);
    v = op == 0 ? v + u : op == 1 ? (u < v ? u : v) : (u > v ? u : v);
  }
  __syncthreads();
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  T r = scratch[0];
  for (int w = 1; w < DL_THREADS / 32; ++w) {
    const T u = scratch[w];
    r = op == 0 ? r + u : op == 1 ? (u < r ? u : r) : (u > r ? u : r);
  }
  return r;
}

// One block per (step, leverage): blockIdx.x = row * G + g.  (Two blocks per SM: 128 registers, no spills.)
__global__ void __launch_bounds__(DL_THREADS, 2)
dice_stats_kernel(const int32_t* __restrict__ hist, const int32_t* __restrict__ bounds, int64_t ld_bounds,
                  const int64_t* __restrict__ offsets, int32_t t_begin, int32_t n_steps,
                  const __grid_constant__ DiceLogs L, int32_t G, double lv0, long long n, long long K, double lw_lo,
                  double lw_hi, double* __restrict__ stats, int32_t* __restrict__ fails) {
  union SelMem {
    struct { unsigned w[4][SEL_BINS]; unsigned c[4][SEL_BINS]; } h;   // weight and cells per bin
    struct { double x[4][SEL_CAP]; unsigned c[4][SEL_CAP]; } g;        // the gathered cells of each target
  };
  __shared__ SelMem U;
  __shared__ double s_lo[4][SEL_LEVELS], s_sc[4][SEL_LEVELS];
  __shared__ int s_bin[4][SEL_LEVELS], s_lvls[4], s_state[4];
  __shared__ long long s_rank[4], s_before[4], s_lt[4], s_eq[4];
  __shared__ unsigned s_ng[4];
  __shared__ double s_ans[4];
  __shared__ double scr_d[DL_THREADS / 32];

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int row = (int)(blockIdx.x / G), g = (int)(blockIdx.x % G), t = t_begin + row;
  const double lu = L.lu[g], ld = L.ld[g], lm = L.lm[g];
  const int amin = bounds[row], amax = bounds[ld_bounds + row];
  const int bmin = bounds[2 * ld_bounds + row], bmax = bounds[3 * ld_bounds + row];
  const int wb = bmax - bmin + 1;
  const int area = (amax - amin + 1) * wb;
  const int32_t* h = hist + offsets[row];
  double* out = stats + ((int64_t)g * n_steps + row) * 12;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);

  if (!isfinite(lu) || !isfinite(ld) || !isfinite(lm)) {
    if (tid == 0) atomicAdd(fails + g, 1);
    if (tid < 12) out[tid] = qnan;
    return;
  }
  // every occupied cell of the box, each thread a fixed strided subset of it: body(x, count)
  auto cells = [&](auto&& body) {
    for (int i = tid; i < area; i += DL_THREADS) {
      const int cnt = h[i];
      if (cnt == 0) continue;
      const int ca = amin + (int)((unsigned)i / (unsigned)wb), cb = bmin + (int)((unsigned)i % (unsigned)wb);
      body(dice_x(lv0, lu, ld, lm, t, ca, cb), cnt);
    }
  };

  // pass 0: the range of x over the occupied cells; the route rule
  double xlo = INFINITY, xhi = -INFINITY;
  cells([&](double x, int) { xlo = fmin(xlo, x); xhi = fmax(xhi, x); });
  xlo = block_reduce(xlo, scr_d, 1);
  xhi = block_reduce(xhi, scr_d, 2);
  if (tid == 0 && !(xlo > lw_lo && xhi < lw_hi)) atomicAdd(fails + g, 1);

  // the select: ranks (n-1)/2, n-K, n-K+(K-1)/2, (n-K-1)/2 of the ascending order
  const long long n_adj = n - K;
  if (tid < 4) {
    const bool ok = tid != 3 || n_adj > 0;
    s_rank[tid] = tid == 0 ? (n - 1) / 2 : tid == 1 ? n - K : tid == 2 ? n - K + (K - 1) / 2 : (n_adj - 1) / 2;
    s_before[tid] = 0;
    s_lvls[tid] = 1;
    s_lo[tid][0] = xlo;
    s_sc[tid][0] = (double)SEL_BINS / (xhi - xlo);
    if (!ok || xlo == xhi) {          // every occupied cell holds the same x
      s_state[tid] = SEL_DONE;
      s_ans[tid] = xlo; s_lt[tid] = 0; s_eq[tid] = n;
    } else {
      s_state[tid] = SEL_ACTIVE;
    }
  }
  __syncthreads();
  for (int level = 0; level < SEL_LEVELS; ++level) {
    bool any = false;
#pragma unroll
    for (int j = 0; j < 4; ++j) any |= s_state[j] == SEL_ACTIVE;
    if (!any) break;
    for (int k = tid; k < 4 * SEL_BINS; k += DL_THREADS) { (&U.h.w[0][0])[k] = 0u; (&U.h.c[0][0])[k] = 0u; }
    __syncthreads();
    cells([&](double x, int cnt) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (s_state[j] != SEL_ACTIVE) continue;
        const int lv = s_lvls[j] - 1;
        bool in = true;
        for (int l = 0; l < lv && in; ++l) in = sel_bin(x, s_lo[j][l], s_sc[j][l]) == s_bin[j][l];
        if (!in) continue;
        const int bin = sel_bin(x, s_lo[j][lv], s_sc[j][lv]);
        atomicAdd(&U.h.w[j][bin], (unsigned)cnt);
        atomicAdd(&U.h.c[j][bin], 1u);
      }
    });
    __syncthreads();
    if (wid < 4 && s_state[wid] == SEL_ACTIVE) {      // warp j: the bin holding target j's rank
      const int j = wid, lv = s_lvls[j] - 1;
      constexpr int per = SEL_BINS / 32;
      long long local = 0;
      for (int k = 0; k < per; ++k) local += U.h.w[j][lane * per + k];
      long long incl = local;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
      }
      const long long want = s_rank[j], excl = incl - local;
      if (want >= excl && want < incl) {
        long long r = want - excl;
        int bin = lane * per;
        for (int k = 0; k < per; ++k) {
          const long long c = U.h.w[j][lane * per + k];
          if (r < c) { bin = lane * per + k; break; }
          r -= c;
        }
        s_bin[j][lv] = bin;
        s_before[j] += want - r;
        s_rank[j] = r;
        if (U.h.c[j][bin] <= (unsigned)SEL_CAP) {
          s_state[j] = SEL_GATHER;
        } else if (lv + 1 < SEL_LEVELS) {
          s_lo[j][lv + 1] = s_lo[j][lv] + (double)bin / s_sc[j][lv];
          s_sc[j][lv + 1] = s_sc[j][lv] * SEL_BINS;
          s_lvls[j] = lv + 2;
        } else {
          s_state[j] = SEL_FAIL;
        }
      }
    }
    __syncthreads();
  }
  // the cells of each target's final bin, ranked one against another
  if (tid < 4) {
    if (s_state[tid] == SEL_ACTIVE) s_state[tid] = SEL_FAIL;
    s_ng[tid] = 0u;
  }
  __syncthreads();
  bool gather = false, failed = false;
#pragma unroll
  for (int j = 0; j < 4; ++j) { gather |= s_state[j] == SEL_GATHER; failed |= s_state[j] == SEL_FAIL; }
  if (failed) {
    if (tid == 0) atomicAdd(fails + g, 1);
    if (tid < 12) out[tid] = qnan;
    return;
  }
  if (gather) {
    cells([&](double x, int cnt) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (s_state[j] != SEL_GATHER) continue;
        bool in = true;
        for (int l = 0; l < s_lvls[j] && in; ++l) in = sel_bin(x, s_lo[j][l], s_sc[j][l]) == s_bin[j][l];
        if (!in) continue;
        const unsigned k = atomicAdd(&s_ng[j], 1u);
        U.g.x[j][k] = x;
        U.g.c[j][k] = (unsigned)cnt;
      }
    });
    __syncthreads();
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
      if (s_state[j] != SEL_GATHER) continue;
      const int m = (int)s_ng[j];
      const long long want = s_rank[j];
      for (int i = tid; i < m; i += DL_THREADS) {
        const double xi = U.g.x[j][i];
        long long lt = 0, eq = 0;
        for (int k = 0; k < m; ++k) {
          const double xk = U.g.x[j][k];
          if (xk < xi) lt += U.g.c[j][k];
          else if (xk == xi) eq += U.g.c[j][k];
        }
        if (lt <= want && want < lt + eq) {     // (equal x: every such lane stores the same)
          s_ans[j] = xi;
          s_lt[j] = s_before[j] + lt;
          s_eq[j] = eq;
        }
      }
    }
    __syncthreads();
  }

  // moments: the top group is every rank >= n - K; cells at the threshold's x split by count
  const double thr = s_ans[1];
  const long long tc_eq = s_lt[1] + s_eq[1] - (n - K);
  double s0 = 0, s1 = 0, s2 = 0;
  int f0 = 0, f1 = 0, f2 = 0;
  cells([&](double x, int cnt) {
    const double v = dice_value(x);
    const long long c = cnt, tc = x > thr ? c : (x == thr ? tc_eq : 0), ac = c - tc;
    s0 += (double)c * v; f0 |= isinf(v);
    if (tc > 0) { s1 += (double)tc * v; f1 |= isinf(v); }
    if (ac > 0) { s2 += (double)ac * v; f2 |= isinf(v); }
  });
  const double size[3] = {(double)n, (double)K, (double)n_adj};
  const double mean[3] = {block_reduce(s0, scr_d, 0) / size[0], block_reduce(s1, scr_d, 0) / size[1],
                          block_reduce(s2, scr_d, 0) / size[2]};
  const int inf_[3] = {__syncthreads_or(f0), __syncthreads_or(f1), __syncthreads_or(f2)};
  double d0 = 0, d1 = 0, d2 = 0, q0 = 0, q1 = 0, q2 = 0;
  cells([&](double x, int cnt) {
    const double v = dice_value(x);
    const long long c = cnt, tc = x > thr ? c : (x == thr ? tc_eq : 0), ac = c - tc;
    const double e0 = v - mean[0];
    d0 += (double)c * fabs(e0);
    q0 += (double)c * (e0 * e0);
    if (tc > 0) {
      const double e = v - mean[1];
      d1 += (double)tc * fabs(e);
      q1 += (double)tc * (e * e);
    }
    if (ac > 0) {
      const double e = v - mean[2];
      d2 += (double)ac * fabs(e);
      q2 += (double)ac * (e * e);
    }
  });
  const double dev[3] = {block_reduce(d0, scr_d, 0), block_reduce(d1, scr_d, 0), block_reduce(d2, scr_d, 0)};
  const double sq[3] = {block_reduce(q0, scr_d, 0), block_reduce(q1, scr_d, 0), block_reduce(q2, scr_d, 0)};

  if (tid == 0) {
    // torch semantics (as rowstats / the tally / the coin lattice): a non-finite member makes mean / MAD / std
    // nan, except that a one-element group's mean is the element itself; an empty adj group is all nan
    double med[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) med[j] = dice_value(s_ans[j]);
    const double single[3] = {med[0], med[1], med[3]};
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      out[0 + j] = mean[j];
      out[3 + j] = dev[j] / size[j];
      out[6 + j] = sqrt(sq[j] / size[j]);
      if (inf_[j]) { out[0 + j] = size[j] == 1 ? single[j] : qnan; out[3 + j] = qnan; out[6 + j] = qnan; }
    }
    out[9] = med[0]; out[10] = med[2]; out[11] = med[3];
    if (n_adj == 0) { out[2] = qnan; out[5] = qnan; out[8] = qnan; out[11] = qnan; }
  }
}

int dice_investors_per_thread(int64_t n) {
  // the fewest that still fit the grid into one wave of four blocks per SM
  const int64_t wave = 4LL * sm_count();
  int R = 1;
  while (R < 4 && (n + (int64_t)DL_THREADS * R - 1) / ((int64_t)DL_THREADS * R) > wave) R *= 2;
  return R;
}

int dice_check_codes(const void* outcomes, int64_t n, int32_t horizon, int64_t ld, int32_t t_begin, int32_t t_end,
                     const char* who) {
  B200_REQUIRE(n >= 1 && n <= INT_MAX && horizon >= 1, "%s: need 1 <= n_investors <= 2^31 - 1, horizon >= 1", who);
  B200_REQUIRE(0 <= t_begin && t_begin < t_end && t_end <= horizon, "%s: need 0 <= t_begin < t_end <= horizon", who);
  B200_REQUIRE(ld >= horizon, "%s: ld_outcomes < horizon", who);
  B200_REQUIRE(outcomes != nullptr, "%s: NULL outcomes", who);
  return 0;
}

}  // namespace b200

using namespace b200;

#define B200_DICE_LAUNCH(KERNEL, ...)                                                      \
  do {                                                                                     \
    if (R == 1) KERNEL<1><<<blocks, DL_THREADS, 0, st>>>(__VA_ARGS__);                     \
    else if (R == 2) KERNEL<2><<<blocks, DL_THREADS, 0, st>>>(__VA_ARGS__);                \
    else KERNEL<4><<<blocks, DL_THREADS, 0, st>>>(__VA_ARGS__);                            \
  } while (0)

extern "C" int b200_dice_lattice_bounds(const void* outcomes, int64_t n_investors, int32_t horizon, int64_t ld_outcomes,
                                        int32_t t_begin, int32_t t_end, int32_t* ab_state, int32_t* bounds,
                                        int64_t ld_bounds, void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  int rc = dice_check_codes(outcomes, n_investors, horizon, ld_outcomes, t_begin, t_end, "dice_lattice_bounds");
  if (rc != 0) return rc;
  B200_REQUIRE(ab_state != nullptr && bounds != nullptr, "dice_lattice_bounds: NULL argument");
  B200_REQUIRE(ld_bounds >= t_end - t_begin, "dice_lattice_bounds: ld_bounds < t_end - t_begin");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t row = (size_t)(t_end - t_begin) * sizeof(int32_t);
  for (int q = 0; q < 4; ++q)    // minima start above any count, maxima at 0 (counts are >= 0)
    B200_CUDA(cudaMemsetAsync(bounds + (int64_t)q * ld_bounds, q % 2 == 0 ? 0x7f : 0, row, st));
  const bool aligned = ((uintptr_t)outcomes & 15) == 0 && ld_outcomes % 16 == 0;
  const int R = dice_investors_per_thread(n_investors);
  const unsigned blocks = (unsigned)((n_investors + (int64_t)DL_THREADS * R - 1) / ((int64_t)DL_THREADS * R));
  B200_DICE_LAUNCH(dice_bounds_kernel, (const uint8_t*)outcomes, n_investors, ld_outcomes, aligned, t_begin, t_end,
                   ab_state, bounds, ld_bounds);
  return check_cuda(cudaGetLastError(), "dice_lattice_bounds launch");
}

extern "C" int b200_dice_lattice_count(const void* outcomes, int64_t n_investors, int32_t horizon, int64_t ld_outcomes,
                                       int32_t t_begin, int32_t t_end, int32_t* ab_state, const int32_t* bounds,
                                       int64_t ld_bounds, const int64_t* offsets, int32_t* hist, int64_t hist_cells,
                                       void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  int rc = dice_check_codes(outcomes, n_investors, horizon, ld_outcomes, t_begin, t_end, "dice_lattice_count");
  if (rc != 0) return rc;
  B200_REQUIRE(ab_state != nullptr && bounds != nullptr && offsets != nullptr && hist != nullptr,
               "dice_lattice_count: NULL argument");
  B200_REQUIRE(ld_bounds >= t_end - t_begin && hist_cells >= 1, "dice_lattice_count: need ld_bounds >= steps, cells >= 1");
  cudaStream_t st = (cudaStream_t)stream;
  B200_CUDA(cudaMemsetAsync(hist, 0, (size_t)hist_cells * sizeof(int32_t), st));
  const bool aligned = ((uintptr_t)outcomes & 15) == 0 && ld_outcomes % 16 == 0;
  const int R = dice_investors_per_thread(n_investors);
  const unsigned blocks = (unsigned)((n_investors + (int64_t)DL_THREADS * R - 1) / ((int64_t)DL_THREADS * R));
  B200_DICE_LAUNCH(dice_count_kernel, (const uint8_t*)outcomes, n_investors, ld_outcomes, aligned, t_begin, t_end,
                   ab_state, bounds, ld_bounds, offsets, hist);
  return check_cuda(cudaGetLastError(), "dice_lattice_count launch");
}

extern "C" int b200_dice_lattice_stats(const int32_t* hist, const int32_t* bounds, int64_t ld_bounds,
                                       const int64_t* offsets, int32_t t_begin, int32_t n_steps, const double* logs_host,
                                       int32_t n_grid, double log_v0, int64_t n_investors, int64_t top, double* stats,
                                       int32_t* fails, void* stream) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(n_grid >= 1 && n_grid <= B200_MAX_GRID, "dice_lattice_stats: n_grid must be in 1..%d", B200_MAX_GRID);
  B200_REQUIRE(t_begin >= 0 && n_steps >= 1 && ld_bounds >= n_steps,
               "dice_lattice_stats: need t_begin >= 0, n_steps >= 1 and ld_bounds >= n_steps");
  B200_REQUIRE(n_investors >= 1 && n_investors <= INT_MAX && top >= 1 && top <= n_investors,
               "dice_lattice_stats: need 1 <= top <= n_investors <= 2^31 - 1");
  B200_REQUIRE(hist != nullptr && bounds != nullptr && offsets != nullptr && logs_host != nullptr && stats != nullptr &&
               fails != nullptr, "dice_lattice_stats: NULL argument");
  DiceLogs L;
  for (int g = 0; g < B200_MAX_GRID; ++g) {
    L.lu[g] = g < n_grid ? logs_host[3 * g] : 0.0;
    L.ld[g] = g < n_grid ? logs_host[3 * g + 1] : 0.0;
    L.lm[g] = g < n_grid ? logs_host[3 * g + 2] : 0.0;
  }
  const double margin = 1e-3;
  const double lw_lo = std::log((double)FLT_MIN) + margin, lw_hi = std::log((double)FLT_MAX) - margin;
  const int64_t blocks = (int64_t)n_grid * n_steps;
  B200_REQUIRE(blocks <= INT_MAX, "dice_lattice_stats: too many (step, leverage) pairs in one call");
  dice_stats_kernel<<<(unsigned)blocks, DL_THREADS, 0, (cudaStream_t)stream>>>(
      hist, bounds, ld_bounds, offsets, t_begin, n_steps, L, n_grid, log_v0, n_investors, top, lw_lo, lw_hi, stats,
      fails);
  return check_cuda(cudaGetLastError(), "dice_lattice_stats launch");
}
