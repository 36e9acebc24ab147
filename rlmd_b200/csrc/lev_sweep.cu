// K1: leverage sweep entry points (b200_lev_sweep / b200_lev_chunk / b200_lev_draw)
// and the kernels that do not depend on the grid-tile templates.
//
// LOG mode (discrete): wealth depends on the outcomes only through their
//   counts, so one warp sweeps one investor row with coalesced 16-byte loads and
//   counts codes with dp4a; HBM-bound, G-independent.
// LOG mode (GBM): running sum of x with its running extremes (to reproduce the
//   reference dtype's overflow/underflow saturation), thread per investor over
//   TMA-staged fp32 tiles, or Philox + Box-Muller draws in registers.
// CHAIN mode kernels live in lev_kernels.cuh / lev_chain_k*.cu.
#include <cstdlib>

#include "lev_kernels.cuh"
#include "tally.cuh"

namespace b200 {

struct LogFactorTable {
  double lm[B200_MAX_OUTCOMES][B200_MAX_GRID];  // log m[k][g]
};
struct LevGrid {
  float lev[B200_MAX_GRID];
};

static int64_t out_ld(const b200_lev_desc& d) { return d.ld_out > 0 ? d.ld_out : d.n_investors; }

template <int K>
__global__ void __launch_bounds__(128)
draw_discrete_kernel(const __grid_constant__ Thresholds th, uint64_t seed, int64_t investor_offset, int32_t H,
                     int64_t N, int64_t ld, uint8_t* __restrict__ out) {
  // one thread per (investor, block of 4 steps)
  const int nblk = (H + 3) >> 2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nblk) return;
  const int64_t row = idx / nblk;
  const int j = (int)(idx - row * nblk);
  const uint64_t id = (uint64_t)(row + investor_offset);
  const Philox4 r = philox4x32_10((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)j, PHILOX_TAG_LEV,
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
  const uint32_t u[4] = {r.x, r.y, r.z, r.w};
  for (int b = 0; b < 4; ++b) {
    const int t = j * 4 + b;
    if (t < H) out[row * ld + t] = (uint8_t)draw_code<K>(u[b], th);
  }
}

// Packed outcomes: four 2-bit codes per byte (step t in byte t>>2, bits 2*(t&3)..+1).
// One thread per (investor, 32-bit word = 16 steps = 4 Philox blocks): the same
// draws as draw_discrete_kernel, packed; steps >= H are written as code 0.
template <int K>
__global__ void __launch_bounds__(128)
draw_discrete_packed_kernel(const __grid_constant__ Thresholds th, uint64_t seed, int64_t investor_offset, int32_t H,
                            int64_t N, int64_t ldb, uint8_t* __restrict__ out) {
  const int nwords = (H + 15) >> 4;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nwords) return;
  const int64_t row = idx / nwords;
  const int w = (int)(idx - row * nwords);
  const uint64_t id = (uint64_t)(row + investor_offset);
  uint32_t word = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int j = w * 4 + q;
    if (j * 4 >= H) break;
    const Philox4 r = philox4x32_10((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)j, PHILOX_TAG_LEV,
                                    (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint32_t u[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int b = 0; b < 4; ++b)
      if (j * 4 + b < H) word |= (uint32_t)draw_code<K>(u[b], th) << (2 * (q * 4 + b));
  }
  uint8_t* dst = out + row * ldb + (int64_t)w * 4;
  if (w * 4 + 4 <= ldb && (((uintptr_t)dst) & 3) == 0) {
    *reinterpret_cast<uint32_t*>(dst) = word;
  } else {
    for (int b = 0; b < 4 && w * 4 + b < ldb; ++b) dst[b] = (uint8_t)(word >> (8 * b));
  }
}

// One bit per flip (the coin: K = 2): step t in byte t >> 3, bit t & 7.  One thread per (investor, 32-bit
// word = 32 steps = 8 Philox blocks): the same draws as draw_discrete_kernel<2>; steps >= H are written 0.
__global__ void __launch_bounds__(128)
draw_discrete_bits1_kernel(const __grid_constant__ Thresholds th, uint64_t seed, int64_t investor_offset, int32_t H,
                           int64_t N, int64_t ldb, uint8_t* __restrict__ out) {
  const int nwords = (H + 31) >> 5;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nwords) return;
  const int64_t row = idx / nwords;
  const int w = (int)(idx - row * nwords);
  const uint64_t id = (uint64_t)(row + investor_offset);
  uint32_t word = 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int j = w * 8 + q;
    if (j * 4 >= H) break;
    const Philox4 r = philox4x32_10((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)j, PHILOX_TAG_LEV,
                                    (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint32_t u[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int b = 0; b < 4; ++b)
      if (j * 4 + b < H) word |= (uint32_t)draw_code<2>(u[b], th) << (q * 4 + b);
  }
  uint8_t* dst = out + row * ldb + (int64_t)w * 4;
  if (w * 4 + 4 <= ldb && (((uintptr_t)dst) & 3) == 0) {
    *reinterpret_cast<uint32_t*>(dst) = word;
  } else {
    for (int b = 0; b < 4 && w * 4 + b < ldb; ++b) dst[b] = (uint8_t)(word >> (8 * b));
  }
}

// uint8 codes -> one bit each: one thread per output word (32 codes)
__global__ void __launch_bounds__(256)
pack_bits1_kernel(const uint8_t* __restrict__ codes, int64_t ld, int32_t H, int64_t N, uint8_t* __restrict__ packed,
                  int64_t ldb) {
  const int nwords = (int)((ldb + 3) >> 2);
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nwords) return;
  const int64_t row = idx / nwords;
  const int w = (int)(idx - row * nwords);
  const uint8_t* __restrict__ src = codes + row * ld + (int64_t)w * 32;
  uint32_t word = 0;
  for (int i = 0; i < 32; ++i) {
    const int t = w * 32 + i;
    if (t < H) word |= (uint32_t)(src[i] & 1u) << i;
  }
  uint8_t* dst = packed + row * ldb + (int64_t)w * 4;
  if (w * 4 + 4 <= ldb && (((uintptr_t)dst) & 3) == 0) {
    *reinterpret_cast<uint32_t*>(dst) = word;
  } else {
    for (int b = 0; b < 4 && w * 4 + b < ldb; ++b) dst[b] = (uint8_t)(word >> (8 * b));
  }
}

// uint8 codes -> packed: one thread per output byte quad (16 codes)
__global__ void __launch_bounds__(256)
pack_codes_kernel(const uint8_t* __restrict__ codes, int64_t ld, int32_t H, int64_t N, uint8_t* __restrict__ packed,
                  int64_t ldb) {
  const int nwords = (int)((ldb + 3) >> 2);   // the pad bytes of a row are written too (zero)
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nwords) return;
  const int64_t row = idx / nwords;
  const int w = (int)(idx - row * nwords);
  const uint8_t* __restrict__ src = codes + row * ld + (int64_t)w * 16;
  uint32_t word = 0;
  if (w * 16 + 16 <= H && (((uintptr_t)src) & 15) == 0) {
    const uint4 v = __ldcs(reinterpret_cast<const uint4*>(src));
    const uint32_t q[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      // four codes, one per byte -> 8 bits
      const uint32_t c = q[i] & 0x03030303u;
      const uint32_t b = (c | (c >> 6) | (c >> 12) | (c >> 18)) & 0xffu;
      word |= b << (8 * i);
    }
  } else {
    for (int i = 0; i < 16; ++i) {
      const int t = w * 16 + i;
      if (t < H) word |= (uint32_t)(src[i] & 3u) << (2 * i);
    }
  }
  uint8_t* dst = packed + row * ldb + (int64_t)w * 4;
  if (w * 4 + 4 <= ldb && (((uintptr_t)dst) & 3) == 0) {
    *reinterpret_cast<uint32_t*>(dst) = word;
  } else {
    for (int b = 0; b < 4 && w * 4 + b < ldb; ++b) dst[b] = (uint8_t)(word >> (8 * b));
  }
}

// ------------------------------------------------ LOG, discrete: counting
// One warp per investor row; lanes stride over 16-byte chunks (coalesced 512 B
// per warp instruction).  Codes 0..3 are counted with dp4a on bit-planes:
//   S1 = sum(code & 1), S2 = sum(code >> 1)   =>   for K <= 3 (codes 0,1,2):
//   n1 = S1, n2 = S2, n0 = H - n1 - n2; K = 4 adds n3 via (code == 3).
template <int K>
__device__ __forceinline__ void count_word(uint32_t wd, uint32_t& s1, uint32_t& s2, uint32_t& s3) {
  s1 = __dp4a(wd & 0x01010101u, 0x01010101u, s1);
  if (K >= 3) s2 = __dp4a((wd >> 1) & 0x01010101u, 0x01010101u, s2);
  if (K >= 4) s3 = __dp4a(wd & (wd >> 1) & 0x01010101u, 0x01010101u, s3);
}

constexpr int COUNT_WARPS = 8;

template <int K>
__global__ void __launch_bounds__(COUNT_WARPS * 32)
log_discrete_stream_kernel(const uint8_t* __restrict__ outcomes, int64_t ld, int32_t H, int64_t N, int32_t G,
                           const __grid_constant__ LogFactorTable lf, double logV0, float* __restrict__ data_T,
                           double* __restrict__ log_w, int32_t* __restrict__ counts, int64_t ldT, const TallyDev tally) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = (int64_t)blockIdx.x * COUNT_WARPS + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * COUNT_WARPS;
  for (int64_t row = warp_global; row < N; row += nwarps) {
    const uint8_t* __restrict__ p = outcomes + row * ld;
    uint32_t s1 = 0, s2 = 0, s3 = 0;
    // head bytes up to 16-byte alignment, body in uint4, tail bytes
    const uintptr_t addr = (uintptr_t)p;
    int head = (int)((16 - (addr & 15)) & 15);
    if (head > H) head = H;
    const int body = (H - head) >> 4;
    const int tail0 = head + (body << 4);
    for (int t = lane; t < head; t += 32) {
      const uint32_t c = p[t];
      s1 += c & 1; if (K >= 3) s2 += (c >> 1) & 1; if (K >= 4) s3 += (c == 3);
    }
    const uint4* __restrict__ q = reinterpret_cast<const uint4*>(p + head);
    int i = lane;
    for (; i + 96 < body; i += 128) {  // 4 independent 16-byte loads in flight per lane
      const uint4 a = __ldcs(q + i), b = __ldcs(q + i + 32), c = __ldcs(q + i + 64), d = __ldcs(q + i + 96);
      count_word<K>(a.x, s1, s2, s3); count_word<K>(a.y, s1, s2, s3);
      count_word<K>(a.z, s1, s2, s3); count_word<K>(a.w, s1, s2, s3);
      count_word<K>(b.x, s1, s2, s3); count_word<K>(b.y, s1, s2, s3);
      count_word<K>(b.z, s1, s2, s3); count_word<K>(b.w, s1, s2, s3);
      count_word<K>(c.x, s1, s2, s3); count_word<K>(c.y, s1, s2, s3);
      count_word<K>(c.z, s1, s2, s3); count_word<K>(c.w, s1, s2, s3);
      count_word<K>(d.x, s1, s2, s3); count_word<K>(d.y, s1, s2, s3);
      count_word<K>(d.z, s1, s2, s3); count_word<K>(d.w, s1, s2, s3);
    }
    for (; i < body; i += 32) {
      const uint4 a = __ldcs(q + i);
      count_word<K>(a.x, s1, s2, s3); count_word<K>(a.y, s1, s2, s3);
      count_word<K>(a.z, s1, s2, s3); count_word<K>(a.w, s1, s2, s3);
    }
    for (int t = tail0 + lane; t < H; t += 32) {
      const uint32_t c = p[t];
      s1 += c & 1; if (K >= 3) s2 += (c >> 1) & 1; if (K >= 4) s3 += (c == 3);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      if (K >= 3) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      if (K >= 4) s3 += __shfl_xor_sync(0xffffffffu, s3, o);
    }
    int n[4];
    if (K == 2) { n[1] = (int)s1; n[0] = H - n[1]; n[2] = n[3] = 0; }
    else if (K == 3) { n[1] = (int)s1; n[2] = (int)s2; n[0] = H - n[1] - n[2]; n[3] = 0; }
    else { n[3] = (int)s3; n[1] = (int)(s1 - s3); n[2] = (int)(s2 - s3); n[0] = H - n[1] - n[2] - n[3]; }
    if (counts != nullptr && lane < K) counts[row * K + lane] = n[lane];
    if (tally.keys != nullptr && lane == 0) tally_insert(tally, tally_key(n[1], n[2], n[3]), 1u);
    if (data_T == nullptr && log_w == nullptr) continue;
    for (int g = lane; g < G; g += 32) {
      double lw = logV0;
#pragma unroll
      for (int k = 0; k < K; ++k)
        if (n[k] > 0) lw += (double)n[k] * lf.lm[k][g];
      if (log_w != nullptr) log_w[(int64_t)g * ldT + row] = lw;
      if (data_T != nullptr) data_T[(int64_t)g * ldT + row] = (float)exp(lw);
    }
  }
}

// ------------------------------------------ LOG, discrete: packed 2-bit codes
// Same contract as log_discrete_stream_kernel on a quarter of the bytes.  The
// masks of a code's low / high bit occupy the even bit positions only, so the
// masks of TWO words share one popc: per 32 codes 2 shifts, 2 LOP3, 2 POPC and
// 2 adds (POPC issues at 16 lanes/clk/SM: ~1/3 of its rate at the HBM rate).
template <int K, int BITS = 2>
__device__ __forceinline__ void count_pair(uint32_t a, uint32_t b, uint32_t& s1, uint32_t& s2, uint32_t& s3) {
  if (BITS == 1) { s1 += __popc(a) + __popc(b); return; }     // one bit per flip: the ones ARE the up moves
  constexpr uint32_t EVEN = 0x55555555u, ODD = 0xaaaaaaaau;
  s1 += __popc((a & EVEN) | ((b << 1) & ODD));
  if (K >= 3) s2 += __popc(((a >> 1) & EVEN) | (b & ODD));
  if (K >= 4) s3 += __popc((a & (a >> 1) & EVEN) | ((b & (b << 1)) & ODD));
}

// Rows that start on a 16-byte boundary (every row of pack_codes / lev_draw) are
// read as whole 16-byte vectors, PACKED_U per lane per iteration, all issued
// before the first is consumed: a 1e4-step row (2500 bytes) is ONE round trip to
// DRAM per warp.  The last vector may reach into the row's pad bytes (ld is a
// multiple of 16 there): the lane that holds it masks the codes of steps >= H.
constexpr int PACKED_U = 6;

template <int BITS>
__device__ __forceinline__ uint32_t word_mask(int valid) {   // low BITS*valid bits, valid clamped to 0..32/BITS
  constexpr int PER = 32 / BITS;
  const int v = min(max(valid, 0), PER);
  return v >= PER ? 0xffffffffu : ((1u << (BITS * v)) - 1u);
}
// mask of a vector whose first `valid` codes are steps < H
template <int BITS>
__device__ __forceinline__ uint4 last_vector_mask(int valid) {
  constexpr int PER = 32 / BITS;
  return make_uint4(word_mask<BITS>(valid), word_mask<BITS>(valid - PER), word_mask<BITS>(valid - 2 * PER),
                    word_mask<BITS>(valid - 3 * PER));
}

// A warp takes 32 consecutive rows: it sweeps them one after the other (every
// lane on the same row: coalesced), lane r keeps the counts of row r, and the
// log-wealth / exp epilogue then runs once for the 32 rows with one row per lane
// - 1/32 of the epilogue instructions per row, uniform (constant-bank) table
// reads and 128-byte coalesced stores of data_T / log_w.
// TALLY: the row's count tuple goes to the tally (tally.cuh) and nothing else is written
// but `counts` - the instantiation the final-time statistics run on.
// BITS = 1: the coin's one-bit-per-flip format (K = 2), half the bytes again.
template <int K, bool TALLY, int BITS = 2>
__global__ void __launch_bounds__(COUNT_WARPS * 32, 4)   // 64 registers: 4 blocks per SM measured best (3: 0.86, 5: 0.83 of HBM)
log_discrete_packed_kernel(const uint8_t* __restrict__ outcomes, int64_t ldb, int32_t H, int64_t N, int32_t G,
                           const __grid_constant__ LogFactorTable lf, double logV0, float* __restrict__ data_T,
                           double* __restrict__ log_w, int32_t* __restrict__ counts, int64_t ldT, const TallyDev tally,
                           int32_t task_rows) {
  if (TALLY) pdl_launch_dependents();   // the compaction's blocks may queue up behind the last wave
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = (int64_t)blockIdx.x * COUNT_WARPS + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * COUNT_WARPS;
  constexpr int PER_BYTE = 8 / BITS;        // codes per byte
  const int nbytes = (H + PER_BYTE - 1) / PER_BYTE;   // bytes that hold codes
  const int full = H / PER_BYTE;            // bytes whose codes are all steps < H
  const int nvec = (nbytes + 15) >> 4;      // 16-byte vectors that hold codes
  const bool vec_rows = (ldb & 15) == 0 && ldb >= (int64_t)nvec * 16;
  // row-invariant shape of the vector walk (see the row loop)
  const int iters = (nvec + 32 * PACKED_U - 1) / (32 * PACKED_U);
  const int rem = nvec - (iters - 1) * 32 * PACKED_U;            // vectors of the last iteration, 1..32*PACKED_U
  const int tail_slots = (rem + 31) >> 5;                        // slots it uses
  const int tail_lanes = rem - (tail_slots - 1) * 32;            // lanes of its last slot, 1..32
  const bool in_tail = lane < tail_lanes;
  // this lane's mask for the last slot: only the row's very last vector holds pad codes
  const uint4 wm = lane == tail_lanes - 1 ? last_vector_mask<BITS>(H - (128 / BITS) * (nvec - 1))
                                          : make_uint4(~0u, ~0u, ~0u, ~0u);
  auto count_byte = [&](int t, uint32_t& s1, uint32_t& s2, uint32_t& s3, const uint8_t* __restrict__ p) {
    uint32_t c = p[t];
    if (t >= full) c &= (1u << (BITS * (H % PER_BYTE))) - 1u;   // the last, partly filled byte
    if (BITS == 1) { s1 += __popc(c); return; }
    s1 += __popc(c & 0x55u);
    if (K >= 3) s2 += __popc((c >> 1) & 0x55u);
    if (K >= 4) s3 += __popc(c & (c >> 1) & 0x55u);
  };
  for (int64_t row0 = warp_global * task_rows; row0 < N; row0 += nwarps * task_rows) {
    const int nr = (int)min((int64_t)task_rows, N - row0);
    uint32_t m1 = 0, m2 = 0, m3 = 0;   // sums of row (row0 + lane)
    for (int r = 0; r < nr; ++r) {
      const uint8_t* __restrict__ p = outcomes + (row0 + r) * ldb;
      uint32_t s1 = 0, s2 = 0, s3 = 0;
      // the next row's lines start their way from DRAM to L2 while this row is counted
      if (r + 1 < nr)
        for (int b = lane * 128; b < nbytes; b += 32 * 128)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(p + ldb + b));
      if (vec_rows && (((uintptr_t)p) & 15) == 0) {
        const uint4* __restrict__ q = reinterpret_cast<const uint4*>(p) + lane;
        // full iterations: PACKED_U vectors per lane, no predicates
        for (int it = 0; it + 1 < iters; ++it, q += 32 * PACKED_U) {
          uint4 v[PACKED_U];
#pragma unroll
          for (int u = 0; u < PACKED_U; ++u) v[u] = __ldcs(q + u * 32);
#pragma unroll
          for (int u = 0; u < PACKED_U; ++u) {
            count_pair<K, BITS>(v[u].x, v[u].y, s1, s2, s3);
            count_pair<K, BITS>(v[u].z, v[u].w, s1, s2, s3);
          }
        }
        // the row's last `rem` vectors: slots below tail_slots-1 are full, slot
        // tail_slots-1 ends at lane tail_lanes-1, whose vector reaches into the pad
        // (everything here but the loaded data was worked out before the row loop)
        uint4 vl = make_uint4(0u, 0u, 0u, 0u);   // the partly filled last slot, kept apart from the array
        if (in_tail) vl = __ldcs(q + (tail_slots - 1) * 32);
        uint4 v[PACKED_U - 1];
#pragma unroll
        for (int u = 0; u < PACKED_U - 1; ++u)
          if (u < tail_slots - 1) v[u] = __ldcs(q + u * 32);
        vl.x &= wm.x; vl.y &= wm.y; vl.z &= wm.z; vl.w &= wm.w;
        count_pair<K, BITS>(vl.x, vl.y, s1, s2, s3);
        count_pair<K, BITS>(vl.z, vl.w, s1, s2, s3);
#pragma unroll
        for (int u = 0; u < PACKED_U - 1; ++u) {
          if (u < tail_slots - 1) {
            count_pair<K, BITS>(v[u].x, v[u].y, s1, s2, s3);
            count_pair<K, BITS>(v[u].z, v[u].w, s1, s2, s3);
          }
        }
      } else {
        // any alignment: head bytes up to 16-byte alignment, body in uint4 (full bytes only), tail bytes
        const uintptr_t addr = (uintptr_t)p;
        int head = (int)((16 - (addr & 15)) & 15);
        if (head > full) head = full;
        const int body = (full - head) >> 4;
        const int tail0 = head + (body << 4);
        for (int t = lane; t < head; t += 32) count_byte(t, s1, s2, s3, p);
        const uint4* __restrict__ q = reinterpret_cast<const uint4*>(p + head);
        for (int i = lane; i < body; i += 32) {
          const uint4 a = __ldcs(q + i);
          count_pair<K, BITS>(a.x, a.y, s1, s2, s3); count_pair<K, BITS>(a.z, a.w, s1, s2, s3);
        }
        for (int t = tail0 + lane; t < nbytes; t += 32) count_byte(t, s1, s2, s3, p);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        if (K >= 3) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        if (K >= 4) s3 += __shfl_xor_sync(0xffffffffu, s3, o);
      }
      if (lane == r) { m1 = s1; m2 = s2; m3 = s3; }
    }
    // ---- epilogue: one row per lane
    // Launched early (B200_LEV_FLAG_EARLY_START), the kernel has only read the outcomes so far; the table and
    // `counts` belong to the previous kernel (the last step's statistics) until it has completed.
    if (TALLY) pdl_wait();
    if (lane < nr) {
      const int64_t row = row0 + lane;
      int n[4];
      if (K == 2) { n[1] = (int)m1; n[0] = H - n[1]; n[2] = n[3] = 0; }
      else if (K == 3) { n[1] = (int)m1; n[2] = (int)m2; n[0] = H - n[1] - n[2]; n[3] = 0; }
      else { n[3] = (int)m3; n[1] = (int)(m1 - m3); n[2] = (int)(m2 - m3); n[0] = H - n[1] - n[2] - n[3]; }
      if (counts != nullptr) {
#pragma unroll
        for (int k = 0; k < K; ++k) counts[row * K + k] = n[k];
      }
      if (TALLY) {
        tally_insert(tally, tally_key(n[1], n[2], n[3]), 1u);
        continue;
      }
      double nd[K];
#pragma unroll
      for (int k = 0; k < K; ++k) nd[k] = (double)n[k];
      for (int g = 0; g < G; ++g) {
        double lw = logV0;
#pragma unroll
        for (int k = 0; k < K; ++k)
          if (n[k] > 0) lw += nd[k] * lf.lm[k][g];
        if (log_w != nullptr) log_w[(int64_t)g * ldT + row] = lw;
        if (data_T != nullptr) data_T[(int64_t)g * ldT + row] = (float)exp(lw);
      }
    }
  }
}

// ----------------------------------------------------------- LOG, GBM
// Saturation of the reference's fp32 chain, decided from the running extremes
// of log-wealth: once the running wealth exceeded FLT_MAX it is inf for good,
// once it fell below half the smallest denormal it is 0 for good.
__device__ __forceinline__ void gbm_finish(double S, double Smax, double Smin, int32_t G,
                                           const LevGrid& lv, double logV0, int64_t row, int64_t ldT,
                                           float* __restrict__ data_T, double* __restrict__ log_w,
                                           bool saturate = true, int64_t state_n = 0) {
  const double LOG_FLT_MAX = 88.72283905206835;    // ln(3.4028234664e38)
  const double LOG_FLT_ZERO = -103.97207708399179; // ln(2^-150)
  if (state_n > 0 && log_w != nullptr) {     // B200_LEV_FLAG_STATE_OUT: the leverage-independent state
    log_w[row] = S; log_w[state_n + row] = Smax; log_w[2 * state_n + row] = Smin;
    log_w = nullptr;
  }
  if (data_T == nullptr && log_w == nullptr) return;
  for (int g = 0; g < G; ++g) {
    const double l = (double)lv.lev[g];
    const double lw = logV0 + l * S;
    const double hi = logV0 + (l >= 0 ? l * Smax : l * Smin);
    const double lo = logV0 + (l >= 0 ? l * Smin : l * Smax);
    if (log_w != nullptr) log_w[(int64_t)g * ldT + row] = lw;
    if (data_T != nullptr) {
      float v;
      if (saturate && hi > LOG_FLT_MAX) v = __int_as_float(0x7f800000);
      else if (saturate && lo < LOG_FLT_ZERO) v = 0.0f;
      else v = (float)exp(lw);
      data_T[(int64_t)g * ldT + row] = v;
    }
  }
}

// 32 steps in fp32 relative to the fp64 base, then fold into the base.
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

template <bool USE_TMA>
__global__ void __launch_bounds__(TILE_ROWS)
log_gbm_stream_kernel(const __grid_constant__ CUtensorMap tmap, const float* __restrict__ x, int64_t ld,
                      const __grid_constant__ LevGrid lv, int32_t H, int64_t N, int32_t G, double logV0,
                      float* __restrict__ data_T, double* __restrict__ log_w, int64_t ldT, bool saturate,
                      int64_t state_n) {
  extern __shared__ __align__(1024) uint8_t tiles[];
  __shared__ __align__(8) uint64_t full[STAGES];
  constexpr int TILE_STEPS = TILE_BYTES / 4;  // 32 floats per row per tile

  const int tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * TILE_ROWS;
  const int ntiles = (H + TILE_STEPS - 1) / TILE_STEPS;

  if (USE_TMA) {
    if (tid == 0) {
      for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
      fence_barrier_init();
    }
    __syncthreads();
    if (tid == 0) {
      const int pre = ntiles < STAGES ? ntiles : STAGES;
      for (int s = 0; s < pre; ++s) {
        mbar_expect_tx(&full[s], TILE_SMEM);
        tma_load_2d(tiles + s * TILE_SMEM, &tmap, &full[s], s * TILE_STEPS, (int)row0);
      }
    }
  }

  GbmAcc acc;
  for (int kt = 0; kt < ntiles; ++kt) {
    const int s = USE_TMA ? kt % STAGES : 0;
    uint8_t* tile = tiles + s * TILE_SMEM;
    if (USE_TMA) {
      mbar_wait(&full[s], (uint32_t)((kt / STAGES) & 1));
    } else {
      __syncthreads();
      const int t0 = kt * TILE_STEPS;
      for (int idx = tid; idx < TILE_ROWS * TILE_STEPS; idx += TILE_ROWS) {
        const int r = idx >> 5, e = idx & 31;
        const int64_t row = row0 + r;
        float v = 0.f;
        if (row < N && t0 + e < H) v = x[row * ld + t0 + e];
        *reinterpret_cast<float*>(tile + swz(r, e >> 2) + (e & 3) * 4) = v;
      }
      __syncthreads();
    }
    const int steps = min(TILE_STEPS, H - kt * TILE_STEPS);
    if (steps == TILE_STEPS) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float4 q = *reinterpret_cast<const float4*>(tile + swz(tid, c));
        acc.step2(q.x, q.y); acc.step2(q.z, q.w);
      }
    } else {
      for (int t = 0; t < steps; ++t)
        acc.step(*reinterpret_cast<const float*>(tile + swz(tid, t >> 2) + (t & 3) * 4));
    }
    acc.fold();
    if (USE_TMA) {
      __syncthreads();
      if (tid == 0 && kt + STAGES < ntiles) {
        mbar_expect_tx(&full[s], TILE_SMEM);
        tma_load_2d(tile, &tmap, &full[s], (kt + STAGES) * TILE_STEPS, (int)row0);
      }
    }
  }
  const int64_t row = row0 + tid;
  if (row < N) gbm_finish(acc.S, acc.Smax, acc.Smin, G, lv, logV0, row, ldT, data_T, log_w, saturate, state_n);
}

// x_t = log_mean + sigma * z_t; four steps per Philox block, two Box-Muller pairs;
// sigma is folded into the radius, the mean into the final FFMA.
__device__ __forceinline__ void gbm_from_words(const Philox4& r, float log_mean, float sigma, float (&x)[4]);
__device__ __forceinline__ void gbm_draw4(uint32_t c0, uint32_t c1, uint32_t j, uint32_t k0, uint32_t k1,
                                          float log_mean, float sigma, float (&x)[4]) {
  gbm_from_words(philox4x32_10(c0, c1, j, PHILOX_TAG_LEV, k0, k1), log_mean, sigma, x);
}
__device__ __forceinline__ void gbm_draw4(uint32_t c0, uint32_t c1, uint32_t j, const PhiloxKeys& K,
                                          float log_mean, float sigma, float (&x)[4]) {
  gbm_from_words(philox4x32_10(c0, c1, j, PHILOX_TAG_LEV, K), log_mean, sigma, x);
}
__device__ __forceinline__ void gbm_from_words(const Philox4& r, float log_mean, float sigma, float (&x)[4]) {
  const float scale2 = box_muller_scale2(sigma);
  float rho, c, s;
  box_muller_polar(r.x, r.y, scale2, rho, c, s);
  x[0] = __fmaf_rn(rho, c, log_mean);
  x[1] = __fmaf_rn(rho, s, log_mean);
  box_muller_polar(r.z, r.w, scale2, rho, c, s);
  x[2] = __fmaf_rn(rho, c, log_mean);
  x[3] = __fmaf_rn(rho, s, log_mean);
}

__global__ void __launch_bounds__(128)
log_gbm_philox_kernel(const __grid_constant__ LevGrid lv, const __grid_constant__ PhiloxKeys K,
                      int64_t investor_offset, float log_mean,
                      float sigma, int32_t H, int64_t N, int32_t G, double logV0, float* __restrict__ data_T,
                      double* __restrict__ log_w, int64_t ldT, bool saturate, int64_t state_n) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= N) return;
  const uint64_t id = (uint64_t)(row + investor_offset);
  const uint32_t c0 = (uint32_t)id, c1 = (uint32_t)(id >> 32);
  GbmAcc acc;
  const int nblk = H >> 2;
  int j = 0;
  for (; j + 8 <= nblk; j += 8) {  // fold every 32 steps
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      float x[4];
      gbm_draw4(c0, c1, (uint32_t)(j + u), K, log_mean, sigma, x);
      acc.step2(x[0], x[1]); acc.step2(x[2], x[3]);
    }
    acc.fold();
  }
  for (; j < nblk; ++j) {
    float x[4];
    gbm_draw4(c0, c1, (uint32_t)j, K, log_mean, sigma, x);
    acc.step2(x[0], x[1]); acc.step2(x[2], x[3]);
  }
  if (H & 3) {
    float x[4];
    gbm_draw4(c0, c1, (uint32_t)nblk, K, log_mean, sigma, x);
    for (int t = 0; t < (H & 3); ++t) acc.step(x[t]);
  }
  acc.fold();
  gbm_finish(acc.S, acc.Smax, acc.Smin, G, lv, logV0, row, ldT, data_T, log_w, saturate, state_n);
}

__global__ void __launch_bounds__(128)
draw_gbm_kernel(uint64_t seed, int64_t investor_offset, float log_mean, float sigma, int32_t H, int64_t N,
                int64_t ld, float* __restrict__ out) {
  const int nblk = (H + 3) >> 2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nblk) return;
  const int64_t row = idx / nblk;
  const int j = (int)(idx - row * nblk);
  const uint64_t id = (uint64_t)(row + investor_offset);
  float x[4];
  gbm_draw4((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)j, (uint32_t)seed, (uint32_t)(seed >> 32), log_mean,
            sigma, x);
  for (int b = 0; b < 4; ++b) {
    const int t = j * 4 + b;
    if (t < H) out[row * ld + t] = x[b];
  }
}

// ------------------------------------------------ GBM series chunk
// Steps [t_begin, t_end) (t_begin a multiple of 32 so that the fp32 partial sums
// fold exactly where the final-time kernels fold them) with the wealth after
// every step dumped: dump[(g*tc + t-t_begin)*N + row].  state = double [5,N]:
// S, its running max and min, then the bit patterns of two 64-bit masks (bit g:
// grid point g's wealth has overflowed / underflowed).  The reference's fp32 chain
// saturates for good in time order - inf once it passes FLT_MAX, 0 once it falls
// below half the smallest denormal, whichever comes first - so the series keeps
// that order per grid point instead of reading it off the running extremes (a path
// that underflowed and later climbed past ln FLT_MAX stays 0).
__device__ __forceinline__ float gbm_wealth(double lw, uint64_t bit, uint64_t& over, uint64_t& under) {
  const double LOG_FLT_MAX = 88.72283905206835;
  const double LOG_FLT_ZERO = -103.97207708399179;
  if (!((over | under) & bit)) {
    if (lw > LOG_FLT_MAX) over |= bit;
    else if (lw < LOG_FLT_ZERO) under |= bit;
  }
  if (over & bit) return __int_as_float(0x7f800000);
  if (under & bit) return 0.0f;
  return (float)exp(lw);
}

template <bool PHILOX>
__global__ void __launch_bounds__(128)
gbm_chunk_kernel(const float* __restrict__ x, int64_t ld, const __grid_constant__ LevGrid lv, uint64_t seed,
                 int64_t investor_offset, float log_mean, float sigma, int32_t t_begin, int32_t t_end, int64_t N,
                 int32_t G, double logV0, double* __restrict__ state, float* __restrict__ dump) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= N) return;
  GbmAcc acc;
  uint64_t over = 0, under = 0;
  if (t_begin > 0) {
    acc.S = state[row]; acc.Smax = state[N + row]; acc.Smin = state[2 * N + row];
    over = (uint64_t)__double_as_longlong(state[3 * N + row]);
    under = (uint64_t)__double_as_longlong(state[4 * N + row]);
  }
  const int64_t tc = t_end - t_begin;
  const uint64_t id = (uint64_t)(row + investor_offset);
  float xb[4];
  for (int t = t_begin; t < t_end; ++t) {
    float xt;
    if (PHILOX) {
      if ((t & 3) == 0 || t == t_begin)
        gbm_draw4((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)(t >> 2), (uint32_t)seed, (uint32_t)(seed >> 32),
                  log_mean, sigma, xb);
      xt = xb[t & 3];
    } else {
      xt = __ldg(x + row * ld + t);
    }
    acc.step(xt);
    const double S = acc.S + (double)acc.p;
    for (int g = 0; g < G; ++g) {
      const float w = gbm_wealth(logV0 + (double)lv.lev[g] * S, 1ull << g, over, under);
      if (dump != nullptr) __stcs(dump + ((int64_t)g * tc + (t - t_begin)) * N + row, w);
    }
    if ((t & 31) == 31) acc.fold();
  }
  acc.fold();
  state[row] = acc.S; state[N + row] = acc.Smax; state[2 * N + row] = acc.Smin;
  state[3 * N + row] = __longlong_as_double((long long)over);
  state[4 * N + row] = __longlong_as_double((long long)under);
}

// ------------------------------------------------------------ host side
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
    else
      cudaGetLastError();
  }
  return fn;
}

int make_row_tile_map(CUtensorMap* map, const void* base, int64_t n_rows, int64_t row_elems, int64_t ld_elems,
                      int elem_bytes) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return set_error(B200_ECUDA, "cuTensorMapEncodeTiled not available from the driver");
  const cuuint64_t dims[2] = {(cuuint64_t)row_elems, (cuuint64_t)n_rows};
  const cuuint64_t strides[1] = {(cuuint64_t)(ld_elems * elem_bytes)};
  const cuuint32_t box[2] = {(cuuint32_t)(TILE_BYTES / elem_bytes), (cuuint32_t)TILE_ROWS};
  const cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = elem_bytes == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  CUresult r = enc(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(B200_ECUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
  return 0;
}

// Steps [t_begin, t_end) of the discrete CHAIN for the whole grid, in tiles of
// <= 32 grid points; each tile re-streams (or re-draws) the outcomes.
// state / dump are laid out for the FULL grid: [G, N] and [G, t_end-t_begin, N].
static int run_chain_discrete(const b200_lev_desc& d, const uint8_t* outcomes, const float* factors_host,
                              int t_begin, int t_end, const float* state_in, float* state_out, float* dump,
                              int64_t ldT, cudaStream_t st) {
  const int64_t N = d.n_investors;
  const int64_t tc = t_end - t_begin;
  for (int g0 = 0; g0 < d.n_grid; g0 += 32) {
    const int g_cnt = d.n_grid - g0 < 32 ? d.n_grid - g0 : 32;
    ChainLaunch a;
    a.d = &d;
    a.outcomes = outcomes;
    for (int k = 0; k < B200_MAX_OUTCOMES; ++k)
      for (int g = 0; g < 32; ++g)
        a.f.m[k][g] = (g < g_cnt && k < d.n_outcomes) ? factors_host[(int64_t)(g0 + g) * d.n_outcomes + k] : 1.0f;
    a.p.t_begin = t_begin;
    a.p.t_end = t_end;
    a.p.G = g_cnt;
    a.p.V0 = d.value_0;
    a.p.N = N;
    a.p.ldT = ldT;
    a.p.state_in = state_in ? state_in + (int64_t)g0 * ldT : nullptr;
    a.p.state_out = state_out + (int64_t)g0 * ldT;
    a.p.dump = dump ? dump + (int64_t)g0 * tc * ldT : nullptr;
    a.variant = d.variant;
    a.st = st;
    int rc;
    switch (d.n_outcomes) {
      case 2: rc = chain_discrete_launch<2>(a); break;
      case 3: rc = chain_discrete_launch<3>(a); break;
      default: rc = chain_discrete_launch<4>(a); break;
    }
    if (rc) return rc;
  }
  return 0;
}

// ------------------------------------------ LOG, discrete: wealth from counts
// Wealth depends on the outcomes only through their counts: a grid of ANY size is
// ONE pass over the outcome array (counts) plus, per tile of 64 grid points, this
// kernel - one thread per investor, the epilogue of the count kernels on its own
// (same expressions in the same order: bit-identical log-wealth and wealth).
template <int K>
__global__ void __launch_bounds__(256)
log_from_counts_kernel(const int32_t* __restrict__ counts, int64_t N, int32_t G,
                       const __grid_constant__ LogFactorTable lf, double logV0, float* __restrict__ data_T,
                       double* __restrict__ log_w, int64_t ldT) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= N) return;
  int n[K];
  double nd[K];
#pragma unroll
  for (int k = 0; k < K; ++k) { n[k] = counts[row * K + k]; nd[k] = (double)n[k]; }
  for (int g = 0; g < G; ++g) {
    double lw = logV0;
#pragma unroll
    for (int k = 0; k < K; ++k)
      if (n[k] > 0) lw += nd[k] * lf.lm[k][g];
    if (log_w != nullptr) log_w[(int64_t)g * ldT + row] = lw;
    if (data_T != nullptr) data_T[(int64_t)g * ldT + row] = (float)exp(lw);
  }
}

static int make_log_table(const b200_lev_desc& d, const float* factors_host, LogFactorTable& lf) {
  for (int k = 0; k < B200_MAX_OUTCOMES; ++k)
    for (int g = 0; g < B200_MAX_GRID; ++g) {
      double v = 0.0;
      if (g < d.n_grid && k < d.n_outcomes) {
        const float m = factors_host[(int64_t)g * d.n_outcomes + k];
        if (m < 0.0f) return set_error(B200_EINVAL, "LOG mode needs factors >= 0 (m[%d][%d] = %g)", g, k, (double)m);
        v = log((double)m);
      }
      lf.lm[k][g] = v;
    }
  return 0;
}

static int run_log_discrete(const b200_lev_desc& d, const uint8_t* outcomes, const float* factors_host,
                            float* data_T, double* log_w, int32_t* counts, const TallyDev& tally, cudaStream_t st) {
  LogFactorTable lf;
  if (factors_host != nullptr) {
    if (int rc = make_log_table(d, factors_host, lf)) return rc;
  } else {
    memset(&lf, 0, sizeof(lf));   // counts / tally only
  }
  const double logV0 = log((double)d.value_0);
  const int64_t N = d.n_investors;
  // a warp per row (uint8 codes) / per 32 rows (packed)
  // rows per packed task (<= 32: one lane per row in the epilogue).  Fewer rows = shorter-lived blocks
  // (kernels on other streams get SM slots sooner) but a thinner epilogue.
  static const int task_rows = [] { const char* e = getenv("B200_PACKED_TASK_ROWS"); int v = e ? atoi(e) : 32;
                                    return v < 1 ? 1 : v > 32 ? 32 : v; }();
  const bool packed = d.outcome_bits == 2 || d.outcome_bits == 1;
  const int64_t warps = packed ? (N + task_rows - 1) / task_rows : N;
  int64_t blocks = (warps + COUNT_WARPS - 1) / COUNT_WARPS;
  // packed: one 32-row task per warp, handed out by the block scheduler (a capped
  // grid would give each warp 3.3 tasks at 1e6 rows: a fifth of the run spent in the tail)
  const int64_t cap = packed ? (int64_t)0x7fffffff : (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  if (packed && tally.keys != nullptr) {   // the tally sink, launched early on request (B200_LEV_FLAG_EARLY_START)
    const auto kern = d.outcome_bits == 1 ? log_discrete_packed_kernel<2, true, 1>
                      : d.n_outcomes == 2 ? log_discrete_packed_kernel<2, true>
                      : d.n_outcomes == 3 ? log_discrete_packed_kernel<3, true>
                                          : log_discrete_packed_kernel<4, true>;
    // All L1, no shared memory: launched early, the kernel's first blocks land on SMs the compaction and the
    // select set up for shared memory, and without this preference the sweep kept that split - a small L1 for
    // its loads in flight - to the end (on B200 the overlapped sweep took 436 us, 409 with it; 387-391 alone).
    B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxL1));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)blocks);
    cfg.blockDim = dim3(COUNT_WARPS * 32);
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    set_pdl_attribute(at[0]);
    cfg.attrs = at;
    cfg.numAttrs = (d.flags & B200_LEV_FLAG_EARLY_START) != 0 && pdl_enabled() ? 1 : 0;
    return check_cuda(cudaLaunchKernelEx(&cfg, kern, outcomes, d.ld_outcomes, d.horizon, N, d.n_grid, lf, logV0, data_T,
                                         log_w, counts, out_ld(d), tally, (int32_t)task_rows),
                      "log_discrete_packed (tally) launch");
  }
#define B200_LOG_LAUNCH(KERNEL, ...)                                                                                  \
  KERNEL<__VA_ARGS__><<<(unsigned)blocks, COUNT_WARPS * 32, 0, st>>>(outcomes, d.ld_outcomes, d.horizon, N, d.n_grid, lf, \
                                                                     logV0, data_T, log_w, counts, out_ld(d), tally B200_EXTRA)
  if (d.outcome_bits == 1) {
#define B200_EXTRA , task_rows
    B200_LOG_LAUNCH(log_discrete_packed_kernel, 2, false, 1);
#undef B200_EXTRA
  } else if (d.outcome_bits == 2) {
#define B200_EXTRA , task_rows
    switch (d.n_outcomes) {
      case 2: B200_LOG_LAUNCH(log_discrete_packed_kernel, 2, false); break;
      case 3: B200_LOG_LAUNCH(log_discrete_packed_kernel, 3, false); break;
      default: B200_LOG_LAUNCH(log_discrete_packed_kernel, 4, false); break;
    }
#undef B200_EXTRA
#define B200_EXTRA
  } else {
    switch (d.n_outcomes) {
      case 2: B200_LOG_LAUNCH(log_discrete_stream_kernel, 2); break;
      case 3: B200_LOG_LAUNCH(log_discrete_stream_kernel, 3); break;
      default: B200_LOG_LAUNCH(log_discrete_stream_kernel, 4); break;
    }
  }
#undef B200_LOG_LAUNCH
#undef B200_EXTRA
  return check_cuda(cudaGetLastError(), "log_discrete_stream launch");
}

static int run_log_gbm(const b200_lev_desc& d, const float* x, const float* lev_host, float* data_T, double* log_w,
                       cudaStream_t st) {
  LevGrid lv;
  for (int g = 0; g < B200_MAX_GRID; ++g) lv.lev[g] = g < d.n_grid ? lev_host[g] : 0.f;
  const double logV0 = log((double)d.value_0);
  const int64_t N = d.n_investors;
  const bool saturate = (d.flags & B200_LEV_FLAG_FINAL_ONLY) == 0;
  const int64_t state_n = (d.flags & B200_LEV_FLAG_STATE_OUT) ? N : 0;
  if (d.source == B200_SRC_PHILOX) {
    const unsigned blocks = (unsigned)((N + 127) / 128);
    log_gbm_philox_kernel<<<blocks, 128, 0, st>>>(lv, philox_keys(d.seed), d.investor_offset, d.log_mean, d.sigma, d.horizon, N,
                                                  d.n_grid, logV0, data_T, log_w, out_ld(d), saturate, state_n);
    return check_cuda(cudaGetLastError(), "log_gbm_philox launch");
  }
  const unsigned blocks = (unsigned)((N + TILE_ROWS - 1) / TILE_ROWS);
  CUtensorMap map;
  memset(&map, 0, sizeof(map));
  if (tma_ok(x, d.ld_outcomes * 4, N)) {
    int rc = make_row_tile_map(&map, x, N, d.horizon, d.ld_outcomes, 4);
    if (rc) return rc;
    auto kern = log_gbm_stream_kernel<true>;
    B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, STAGES * TILE_SMEM));
    kern<<<blocks, TILE_ROWS, STAGES * TILE_SMEM, st>>>(map, x, d.ld_outcomes, lv, d.horizon, N, d.n_grid, logV0,
                                                        data_T, log_w, out_ld(d), saturate, state_n);
  } else {
    log_gbm_stream_kernel<false><<<blocks, TILE_ROWS, TILE_SMEM, st>>>(map, x, d.ld_outcomes, lv, d.horizon, N,
                                                                       d.n_grid, logV0, data_T, log_w, out_ld(d), saturate, state_n);
  }
  return check_cuda(cudaGetLastError(), "log_gbm_stream launch");
}

int chain_stages() {
  static int v = [] {
    const char* e = getenv("B200_CHAIN_STAGES");
    int x = e ? atoi(e) : 2;
    return x < 1 ? 1 : x > STAGES ? STAGES : x;
  }();
  return v;
}

static int validate(const b200_lev_desc* d) {
  B200_REQUIRE(d != nullptr, "lev: desc is NULL");
  B200_REQUIRE(d->n_investors >= 0 && d->n_investors < ((int64_t)1 << 40), "lev: n_investors out of range");
  B200_REQUIRE(d->horizon >= 1, "lev: horizon must be >= 1");
  B200_REQUIRE(d->ld_out == 0 || d->ld_out >= d->n_investors, "lev: ld_out < n_investors");
  B200_REQUIRE(d->n_grid >= 1 && d->n_grid <= B200_MAX_GRID, "lev: n_grid must be in 1..%d", B200_MAX_GRID);
  B200_REQUIRE(d->kind == B200_LEV_DISCRETE || d->kind == B200_LEV_GBM, "lev: unknown kind %d", d->kind);
  B200_REQUIRE(d->source == B200_SRC_STREAM || d->source == B200_SRC_PHILOX, "lev: unknown source %d", d->source);
  B200_REQUIRE(d->variant >= 0 && d->variant <= 3, "lev: variant must be 0 (auto), 1 (FSEL), 2 (LDS) or 3 (FMA)");
  if (d->kind == B200_LEV_DISCRETE) {
    B200_REQUIRE(d->n_outcomes >= 2 && d->n_outcomes <= B200_MAX_OUTCOMES, "lev: n_outcomes must be in 2..%d",
                 B200_MAX_OUTCOMES);
    if (d->source == B200_SRC_PHILOX)
      for (int k = 1; k < d->n_outcomes - 1; ++k)
        B200_REQUIRE(d->thresholds[k] >= d->thresholds[k - 1], "lev: thresholds must ascend");
  }
  B200_REQUIRE(d->outcome_bits == 0 || d->outcome_bits == 8 || d->outcome_bits == 2 || d->outcome_bits == 1,
               "lev: outcome_bits must be 0/8 (uint8 codes), 2 (packed) or 1 (packed coin)");
  if (d->outcome_bits == 2) {
    B200_REQUIRE(d->kind == B200_LEV_DISCRETE, "lev: packed outcomes are discrete codes");
    B200_REQUIRE(d->ld_outcomes >= ((int64_t)d->horizon + 3) / 4, "lev: packed ld_outcomes (bytes) < ceil(horizon/4)");
  } else if (d->outcome_bits == 1) {
    B200_REQUIRE(d->kind == B200_LEV_DISCRETE && d->n_outcomes == 2, "lev: one-bit outcomes are the coin's (K = 2)");
    B200_REQUIRE(d->ld_outcomes >= ((int64_t)d->horizon + 7) / 8, "lev: packed ld_outcomes (bytes) < ceil(horizon/8)");
  } else if (d->source == B200_SRC_STREAM) {
    B200_REQUIRE(d->ld_outcomes >= d->horizon, "lev: ld_outcomes < horizon");
  }
  return 0;
}

}  // namespace b200

using namespace b200;

extern "C" int b200_lev_sweep(const b200_lev_desc* desc, const void* outcomes, const float* factors, float* data_T,
                              double* log_w, int32_t* counts, void* stream) {
  int rc = validate(desc);
  if (rc) return rc;
  const b200_lev_desc& d = *desc;
  cudaStream_t st = (cudaStream_t)stream;
  B200_REQUIRE(factors != nullptr, "lev_sweep: factors is NULL");
  B200_REQUIRE(d.source == B200_SRC_PHILOX || outcomes != nullptr || d.n_investors == 0,
               "lev_sweep: outcomes is NULL for a streamed sweep");
  if (d.n_investors == 0) return 0;

  // the tiny factor table travels as a kernel parameter
  const float* host_f = factors;

  if (d.kind == B200_LEV_DISCRETE) {
    if (d.mode == B200_MODE_CHAIN) {
      B200_REQUIRE(data_T != nullptr, "lev_sweep: CHAIN mode needs data_T");
      B200_REQUIRE((d.outcome_bits != 2 && d.outcome_bits != 1) || d.source == B200_SRC_PHILOX,
                   "lev_sweep: the CHAIN kernels take uint8 codes (packed outcomes feed the LOG sweep)");
      return run_chain_discrete(d, (const uint8_t*)outcomes, host_f, 0, d.horizon, nullptr, data_T, nullptr, out_ld(d), st);
    }
    if (d.mode == B200_MODE_LOG) {
      B200_REQUIRE(d.source == B200_SRC_STREAM, "lev_sweep: discrete LOG mode takes streamed outcomes");
      B200_REQUIRE(data_T || log_w || counts, "lev_sweep: LOG mode needs at least one output");
      return run_log_discrete(d, (const uint8_t*)outcomes, host_f, data_T, log_w, counts, TallyDev{nullptr, nullptr, nullptr, 0}, st);
    }
    return set_error(B200_EINVAL, "lev_sweep: unknown mode %d", d.mode);
  }
  B200_REQUIRE(d.mode == B200_MODE_LOG, "lev_sweep: GBM runs in LOG mode only (expf chains are not reproducible)");
  B200_REQUIRE(data_T || log_w, "lev_sweep: LOG mode needs at least one output");
  return run_log_gbm(d, (const float*)outcomes, host_f, data_T, log_w, st);
}

extern "C" int b200_lev_tally(const b200_lev_desc* desc, const void* outcomes, const b200_tally_plan* plan,
                              void* workspace, int32_t* counts, void* stream) {
  int rc = validate(desc);
  if (rc) return rc;
  const b200_lev_desc& d = *desc;
  B200_REQUIRE(d.kind == B200_LEV_DISCRETE && d.source == B200_SRC_STREAM,
               "lev_tally: discrete sweeps over streamed outcomes only");
  B200_REQUIRE(plan != nullptr && d.n_investors <= plan->rows_cap, "lev_tally: more rows than the plan's rows_cap");
  TallyDev t;
  if ((rc = tally_device_view(plan, workspace, d.horizon, &t))) return rc;
  if (d.n_investors == 0) return 0;
  B200_REQUIRE(outcomes != nullptr, "lev_tally: outcomes is NULL");
  return run_log_discrete(d, (const uint8_t*)outcomes, nullptr, nullptr, nullptr, counts, t, (cudaStream_t)stream);
}

extern "C" int b200_lev_draw(const b200_lev_desc* desc, void* out, void* stream) {
  int rc = validate(desc);
  if (rc) return rc;
  const b200_lev_desc& d = *desc;
  cudaStream_t st = (cudaStream_t)stream;
  B200_REQUIRE(out != nullptr || d.n_investors == 0, "lev_draw: out is NULL");
  if (d.n_investors == 0) return 0;
  if (d.outcome_bits == 1) {
    const int64_t words = d.n_investors * (int64_t)((d.horizon + 31) >> 5);
    const unsigned pb = (unsigned)((words + 127) / 128);
    Thresholds th;
    for (int k = 0; k < B200_MAX_OUTCOMES; ++k) th.t[k] = d.thresholds[k];
    draw_discrete_bits1_kernel<<<pb, 128, 0, st>>>(th, d.seed, d.investor_offset, d.horizon, d.n_investors,
                                                   d.ld_outcomes, (uint8_t*)out);
    return check_cuda(cudaGetLastError(), "lev_draw (one bit) launch");
  }
  if (d.outcome_bits == 2) {
    const int64_t words = d.n_investors * (int64_t)((d.horizon + 15) >> 4);
    const unsigned pb = (unsigned)((words + 127) / 128);
    Thresholds th;
    for (int k = 0; k < B200_MAX_OUTCOMES; ++k) th.t[k] = d.thresholds[k];
    switch (d.n_outcomes) {
      case 2: draw_discrete_packed_kernel<2><<<pb, 128, 0, st>>>(th, d.seed, d.investor_offset, d.horizon,
                                                                 d.n_investors, d.ld_outcomes, (uint8_t*)out); break;
      case 3: draw_discrete_packed_kernel<3><<<pb, 128, 0, st>>>(th, d.seed, d.investor_offset, d.horizon,
                                                                 d.n_investors, d.ld_outcomes, (uint8_t*)out); break;
      default: draw_discrete_packed_kernel<4><<<pb, 128, 0, st>>>(th, d.seed, d.investor_offset, d.horizon,
                                                                  d.n_investors, d.ld_outcomes, (uint8_t*)out); break;
    }
    return check_cuda(cudaGetLastError(), "lev_draw (packed) launch");
  }
  B200_REQUIRE(d.ld_outcomes >= d.horizon, "lev_draw: ld_outcomes < horizon");
  const int64_t work = d.n_investors * (int64_t)((d.horizon + 3) >> 2);
  const unsigned blocks = (unsigned)((work + 127) / 128);
  if (d.kind == B200_LEV_GBM) {
    draw_gbm_kernel<<<blocks, 128, 0, st>>>(d.seed, d.investor_offset, d.log_mean, d.sigma, d.horizon,
                                            d.n_investors, d.ld_outcomes, (float*)out);
  } else {
    Thresholds th;
    for (int k = 0; k < B200_MAX_OUTCOMES; ++k) th.t[k] = d.thresholds[k];
    switch (d.n_outcomes) {
      case 2: draw_discrete_kernel<2><<<blocks, 128, 0, st>>>(th, d.seed, d.investor_offset, d.horizon,
                                                              d.n_investors, d.ld_outcomes, (uint8_t*)out); break;
      case 3: draw_discrete_kernel<3><<<blocks, 128, 0, st>>>(th, d.seed, d.investor_offset, d.horizon,
                                                              d.n_investors, d.ld_outcomes, (uint8_t*)out); break;
      default: draw_discrete_kernel<4><<<blocks, 128, 0, st>>>(th, d.seed, d.investor_offset, d.horizon,
                                                               d.n_investors, d.ld_outcomes, (uint8_t*)out); break;
    }
  }
  return check_cuda(cudaGetLastError(), "lev_draw launch");
}

extern "C" int b200_lev_from_counts(const b200_lev_desc* desc, const int32_t* counts, const float* factors,
                                    float* data_T, double* log_w, void* stream) {
  int rc = validate(desc);
  if (rc) return rc;
  const b200_lev_desc& d = *desc;
  B200_REQUIRE(d.kind == B200_LEV_DISCRETE, "lev_from_counts: discrete sweeps only");
  B200_REQUIRE(factors != nullptr, "lev_from_counts: factors is NULL");
  B200_REQUIRE(data_T || log_w, "lev_from_counts: needs at least one output");
  if (d.n_investors == 0) return 0;
  B200_REQUIRE(counts != nullptr, "lev_from_counts: counts is NULL");
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  LogFactorTable lf;
  if ((rc = make_log_table(d, factors, lf))) return rc;
  const double logV0 = log((double)d.value_0);
  const int64_t N = d.n_investors;
  const unsigned blocks = (unsigned)((N + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  switch (d.n_outcomes) {
    case 2: log_from_counts_kernel<2><<<blocks, 256, 0, st>>>(counts, N, d.n_grid, lf, logV0, data_T, log_w, out_ld(d)); break;
    case 3: log_from_counts_kernel<3><<<blocks, 256, 0, st>>>(counts, N, d.n_grid, lf, logV0, data_T, log_w, out_ld(d)); break;
    default: log_from_counts_kernel<4><<<blocks, 256, 0, st>>>(counts, N, d.n_grid, lf, logV0, data_T, log_w, out_ld(d)); break;
  }
  return check_cuda(cudaGetLastError(), "lev_from_counts launch");
}

extern "C" int b200_lev_pack(const uint8_t* codes, int64_t n_investors, int32_t horizon, int64_t ld_codes,
                             uint8_t* packed, int64_t ld_packed, void* stream) {
  return b200_lev_pack_bits(codes, n_investors, horizon, ld_codes, packed, ld_packed, 2, stream);
}

extern "C" int b200_lev_pack_bits(const uint8_t* codes, int64_t n_investors, int32_t horizon, int64_t ld_codes,
                                  uint8_t* packed, int64_t ld_packed, int32_t bits, void* stream) {
  B200_REQUIRE(n_investors >= 0 && horizon >= 1, "lev_pack: need n_investors >= 0 and horizon >= 1");
  B200_REQUIRE(bits == 1 || bits == 2, "lev_pack: bits must be 1 or 2");
  if (n_investors == 0) return 0;
  B200_REQUIRE(codes != nullptr && packed != nullptr, "lev_pack: NULL buffer");
  B200_REQUIRE(ld_codes >= horizon, "lev_pack: ld_codes < horizon");
  if (bits == 1) {
    B200_REQUIRE(ld_packed >= ((int64_t)horizon + 7) / 8, "lev_pack: ld_packed < ceil(horizon/8)");
    const int64_t words = n_investors * ((ld_packed + 3) >> 2);
    const int64_t blocks = (words + 255) / 256;
    B200_REQUIRE(blocks <= 0x7fffffff, "lev_pack: too many rows for one launch");
    pack_bits1_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(codes, ld_codes, horizon, n_investors, packed,
                                                                           ld_packed);
    return check_cuda(cudaGetLastError(), "lev_pack launch");
  }
  B200_REQUIRE(ld_packed >= ((int64_t)horizon + 3) / 4, "lev_pack: ld_packed < ceil(horizon/4)");
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  const int64_t words = n_investors * ((ld_packed + 3) >> 2);
  const int64_t blocks = (words + 255) / 256;
  B200_REQUIRE(blocks <= 0x7fffffff, "lev_pack: too many rows for one launch");
  pack_codes_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(codes, ld_codes, horizon, n_investors, packed,
                                                                         ld_packed);
  return check_cuda(cudaGetLastError(), "lev_pack launch");
}

extern "C" int b200_lev_chunk(const b200_lev_desc* desc, const void* outcomes, const float* factors, int32_t t_begin,
                              int32_t t_end, void* state, float* dump, void* stream) {
  int rc = validate(desc);
  if (rc) return rc;
  const b200_lev_desc& d = *desc;
  cudaStream_t st = (cudaStream_t)stream;
  B200_REQUIRE(factors != nullptr && state != nullptr, "lev_chunk: factors/state is NULL");
  B200_REQUIRE(0 <= t_begin && t_begin < t_end && t_end <= d.horizon, "lev_chunk: need 0 <= t_begin < t_end <= horizon");
  B200_REQUIRE(d.source == B200_SRC_PHILOX || outcomes != nullptr || d.n_investors == 0,
               "lev_chunk: outcomes is NULL for a streamed sweep");
  if (d.n_investors == 0) return 0;
  if (d.kind == B200_LEV_DISCRETE) {
    B200_REQUIRE(d.mode == B200_MODE_CHAIN, "lev_chunk: discrete chunks run in CHAIN mode");
    B200_REQUIRE((d.outcome_bits != 2 && d.outcome_bits != 1) || d.source == B200_SRC_PHILOX,
                 "lev_chunk: the CHAIN kernels take uint8 codes");
    B200_REQUIRE(d.source != B200_SRC_PHILOX || (t_begin & 3) == 0, "lev_chunk: Philox chunks start at a multiple of 4");
    float* stf = (float*)state;
    return run_chain_discrete(d, (const uint8_t*)outcomes, factors, t_begin, t_end, t_begin > 0 ? stf : nullptr, stf,
                              dump, d.n_investors, st);
  }
  B200_REQUIRE((t_begin & 31) == 0, "lev_chunk: GBM chunks start at a multiple of 32");
  LevGrid lv;
  for (int g = 0; g < B200_MAX_GRID; ++g) lv.lev[g] = g < d.n_grid ? factors[g] : 0.f;
  const double logV0 = log((double)d.value_0);
  const unsigned blocks = (unsigned)((d.n_investors + 127) / 128);
  if (d.source == B200_SRC_PHILOX)
    gbm_chunk_kernel<true><<<blocks, 128, 0, st>>>(nullptr, 0, lv, d.seed, d.investor_offset, d.log_mean, d.sigma,
                                                   t_begin, t_end, d.n_investors, d.n_grid, logV0, (double*)state, dump);
  else
    gbm_chunk_kernel<false><<<blocks, 128, 0, st>>>((const float*)outcomes, d.ld_outcomes, lv, d.seed,
                                                    d.investor_offset, d.log_mean, d.sigma, t_begin, t_end,
                                                    d.n_investors, d.n_grid, logV0, (double*)state, dump);
  return check_cuda(cudaGetLastError(), "gbm_chunk launch");
}


// ------------------------------------------------ GBM: valid runs per grid point from the state
namespace b200 {
constexpr int VALID_TILE = 16;     // grid points per sweep of the state

__global__ void __launch_bounds__(256)
gbm_valid_kernel(const double* __restrict__ state, const float* __restrict__ data_T, int64_t ldT, int64_t N,
                 const __grid_constant__ LevGrid lv, int32_t G, double logV0, double* __restrict__ out) {
  __shared__ double red_d[32];
  __shared__ long long red_i[32];
  const double LOG_FLT_MAX = 88.72283905206835, LOG_FLT_ZERO = -103.97207708399179;
  for (int g0 = 0; g0 < G; g0 += VALID_TILE) {
    double sum[VALID_TILE];
    int cnt[VALID_TILE];            // a thread sees far fewer than 2^31 runs
#pragma unroll
    for (int q = 0; q < VALID_TILE; ++q) { sum[q] = 0.0; cnt[q] = 0; }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
      const double S = __ldcs(state + i);
      if (data_T != nullptr) {          // the sweep's own fp32 wealth decides
        float w[VALID_TILE];
#pragma unroll
        for (int q = 0; q < VALID_TILE; ++q)
          w[q] = g0 + q < G ? __ldcs(data_T + (int64_t)(g0 + q) * ldT + i) : 0.0f;
#pragma unroll
        for (int q = 0; q < VALID_TILE; ++q)
          if (w[q] > 0.0f && w[q] < __int_as_float(0x7f800000)) { sum[q] += S; ++cnt[q]; }
        continue;
      }
      const double Smax = state[N + i], Smin = state[2 * N + i];
#pragma unroll
      for (int q = 0; q < VALID_TILE; ++q) {
        if (g0 + q >= G) break;
        const double l = (double)lv.lev[g0 + q];
        const double hi = logV0 + (l >= 0 ? l * Smax : l * Smin);
        const double lo = logV0 + (l >= 0 ? l * Smin : l * Smax);
        bool ok = !(hi > LOG_FLT_MAX) && !(lo < LOG_FLT_ZERO);
        if (ok) { const float x = (float)exp(logV0 + l * S); ok = x > 0.0f && x < __int_as_float(0x7f800000); }
        if (ok) { sum[q] += S; ++cnt[q]; }
      }
    }
#pragma unroll
    for (int q = 0; q < VALID_TILE; ++q) {
      if (g0 + q >= G) break;
      const double s = block_sum(sum[q], red_d);
      const long long c = block_sum((long long)cnt[q], red_i);
      if (threadIdx.x == 0) {
        atomicAdd(out + 2 * (g0 + q), (double)c);      // counts < 2^53: exact in fp64
        atomicAdd(out + 2 * (g0 + q) + 1, s);
      }
    }
  }
}

// Growth-rate summaries of the whole grid from the statistics of S (one row) and the valid-run sums:
// g = l S / H, so mean / std / extremes / quantiles scale with l / H (the q-quantile of a row with
// l < 0 is l / H times S's (1-q)-quantile: Hyndman-Fan type 8 is symmetric).
//   base  : the b200_growth_summary row of S with log_v0 = 0, H = 1: [valid, mean, std, mean_valid,
//           min, max, then the quantiles `need[0..n_need)` of S]
//   valid : [G,2] from b200_gbm_valid (all-reduced over ranks by the caller)
//   out   : [G, 6 + n_q]
__global__ void gbm_assemble_kernel(const double* __restrict__ base, const double* __restrict__ valid,
                                    const __grid_constant__ LevGrid lv, int32_t G, double H, int32_t n_q,
                                    const int32_t* __restrict__ pick_pos, const int32_t* __restrict__ pick_neg,
                                    double* __restrict__ out) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const double l = (double)lv.lev[g] / H;
  const bool pos = l >= 0;
  double* o = out + (int64_t)g * (6 + n_q);
  const double cnt = valid[2 * g], sv = valid[2 * g + 1];
  o[0] = cnt;
  o[1] = l * base[1];
  o[2] = fabs(l) * base[2];
  o[3] = cnt > 0 ? l * sv / cnt : __longlong_as_double(0x7ff8000000000000LL);
  o[4] = pos ? l * base[4] : l * base[5];
  o[5] = pos ? l * base[5] : l * base[4];
  for (int q = 0; q < n_q; ++q) o[6 + q] = l * base[6 + (pos ? pick_pos[q] : pick_neg[q])];
}
}  // namespace b200

extern "C" int b200_gbm_valid(const double* state, const float* data_T, int64_t n, int64_t ld_T, const float* lev_host,
                              int32_t n_grid, double log_v0, double* out, void* stream) {
  B200_REQUIRE(n >= 0 && n_grid >= 1 && n_grid <= B200_MAX_GRID, "gbm_valid: need n >= 0 and 1 <= n_grid <= %d", B200_MAX_GRID);
  B200_REQUIRE(lev_host != nullptr && out != nullptr, "gbm_valid: NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  B200_CUDA(cudaMemsetAsync(out, 0, (size_t)n_grid * 2 * sizeof(double), st));
  if (n == 0) return 0;
  B200_REQUIRE(state != nullptr, "gbm_valid: state is NULL");
  B200_REQUIRE(data_T == nullptr || ld_T >= n, "gbm_valid: ld_T < n");
  LevGrid lv;
  for (int g = 0; g < B200_MAX_GRID; ++g) lv.lev[g] = g < n_grid ? lev_host[g] : 0.f;
  const int64_t want = (n + 255) / 256;
  const unsigned blocks = (unsigned)(want < (int64_t)sm_count() * 16 ? want : (int64_t)sm_count() * 16);
  gbm_valid_kernel<<<blocks, 256, 0, st>>>(state, data_T, ld_T, n, lv, n_grid, log_v0, out);
  return check_cuda(cudaGetLastError(), "gbm_valid launch");
}

extern "C" int b200_gbm_growth_assemble(const double* base_row, const double* valid, const float* lev_host,
                                        int32_t n_grid, int32_t horizon, int32_t n_q, const int32_t* pick_pos,
                                        const int32_t* pick_neg, double* out, void* stream) {
  B200_REQUIRE(n_grid >= 1 && n_grid <= B200_MAX_GRID && horizon >= 1 && n_q >= 0, "gbm_growth_assemble: bad sizes");
  B200_REQUIRE(base_row && valid && lev_host && out && (n_q == 0 || (pick_pos && pick_neg)),
               "gbm_growth_assemble: NULL argument");
  LevGrid lv;
  for (int g = 0; g < B200_MAX_GRID; ++g) lv.lev[g] = g < n_grid ? lev_host[g] : 0.f;
  gbm_assemble_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(base_row, valid, lv, n_grid, (double)horizon, n_q, pick_pos,
                                                          pick_neg, out);
  return check_cuda(cudaGetLastError(), "gbm_growth_assemble launch");
}
