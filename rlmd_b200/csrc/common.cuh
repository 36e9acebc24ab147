// Shared device/host helpers for the rlmd_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>

#include "../../include/rlmd_b200.h"

namespace b200 {

// ----------------------------------------------------------------- errors
int set_error(int code, const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

#define B200_CUDA(expr)                                   \
  do {                                                    \
    int _rc = ::b200::check_cuda((expr), #expr);          \
    if (_rc != 0) return _rc;                             \
  } while (0)

#define B200_REQUIRE(cond, ...)                                     \
  do {                                                              \
    if (!(cond)) return ::b200::set_error(B200_EINVAL, __VA_ARGS__); \
  } while (0)

int sm_count();

// -------------------------------------------- programmatic dependent launch
// A kernel launched with the programmatic-stream-serialization attribute may start once every block of the
// stream's previous kernel has executed launch_dependents (or exited); its griddepcontrol.wait then blocks
// until that kernel has completed and its memory is visible.  Both instructions are no-ops in a kernel
// launched without the attribute.  B200_PDL=0 in the environment (read once) launches without it.
bool pdl_enabled();
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
inline void set_pdl_attribute(cudaLaunchAttribute& a) {
  a.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  a.val.programmaticStreamSerializationAllowed = 1;
}

// ------------------------------------------------------------ Philox4x32-10
// Counter-based generator (Salmon et al., SC'11).  Words are consumed as
//   counter = (investor_id lo, investor_id hi, block index, stream tag)
//   key     = (seed lo, seed hi)
// so a draw depends only on (seed, global investor id, time block): results
// are independent of the GPU count and of the launch geometry.
struct Philox4 {
  uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2,
                                                           uint32_t c3, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  const uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0;
    c1 = lo1;
    c2 = n2;
    c3 = lo0;
    k0 += W0;
    k1 += W1;
  }
  return Philox4{c0, c1, c2, c3};
}

// The ten round keys (k + r * Weyl constant) formed once on the host and handed
// to a kernel as a parameter: the rounds then read them straight from the
// constant bank instead of re-deriving them with uniform-datapath adds, which
// cost issue slots in the generator-bound sweeps.
struct PhiloxKeys {
  uint32_t k0[10], k1[10];
};
inline PhiloxKeys philox_keys(uint64_t seed) {
  PhiloxKeys K;
  uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32);
  for (int r = 0; r < 10; ++r) {
    K.k0[r] = a;
    K.k1[r] = b;
    a += 0x9E3779B9u;
    b += 0xBB67AE85u;
  }
  return K;
}
__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 const PhiloxKeys& K) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    const uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    const uint32_t n0 = hi1 ^ c1 ^ K.k0[r];
    const uint32_t n2 = hi0 ^ c3 ^ K.k1[r];
    c0 = n0;
    c1 = lo1;
    c2 = n2;
    c3 = lo0;
  }
  return Philox4{c0, c1, c2, c3};
}

enum : uint32_t {
  PHILOX_TAG_LEV = 0x4C455600u,   // 'LEV'
  PHILOX_TAG_ENV = 0x454E5600u,   // 'ENV'
  PHILOX_TAG_REPLAY = 0x52504C00u // 'RPL'
};

// Box-Muller on two uniform words, 12 instructions per pair of normals (4 MUFU):
//   u1    = fl32(fl32(a) * 2^-32 + 2^-33)        in (0, 1]   (one I2F, one FFMA)
//   theta = fl32(int32(b)) * pi * 2^-31          in [-pi, pi] (one I2F, one FMUL)
//   rho   = sqrt(scale2 * log2(u1)),  scale2 = -2 ln2 * sigma^2   (lg2/sqrt.approx)
//   y0 = rho cos(theta), y1 = rho sin(theta)      ~ N(0, sigma^2)
// oracle/philox_oracle.py:gbm_returns restates exactly this.
__device__ __forceinline__ float box_muller_scale2(float sigma) { return -1.3862943611198906f * sigma * sigma; }
__device__ __forceinline__ void box_muller_polar(uint32_t a, uint32_t b, float scale2, float& rho, float& c,
                                                 float& s) {
  const float u1 = __fmaf_rn(__uint2float_rn(a), 2.3283064365386963e-10f, 1.1641532182693481e-10f);
  float l2;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(u1));
  const float q = __fmul_rn(l2, scale2);
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rho) : "f"(q));
  const float th = __fmul_rn(__int2float_rn((int32_t)b), 1.4629180792671596e-09f);  // pi * 2^-31
  s = __sinf(th);
  c = __cosf(th);
}
// Unit normals.
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
  float rho, c, s;
  box_muller_polar(a, b, -1.3862943611198906f, rho, c, s);
  z0 = rho * c;
  z1 = rho * s;
}

// np.sum / np.mean of a contiguous fp64 vector: NumPy's pairwise_sum
// (numpy/core/src/umath/loops_utils.h.src) for n <= PW_BLOCKSIZE (128) - plain
// left-to-right below 8 elements, 8 running partial sums from 8 on.  The envs'
// exact-equality termination tests need the reference's summation order.
// NG > 0: n == NG is a compile-time constant (the short form unrolls).
template <int NG = 0, typename F>
__device__ __forceinline__ double np_sum(int n, F term) {
  if (NG > 0 ? NG < 8 : n < 8) {
    double res = term(0);
    if (NG > 0) {
#pragma unroll
      for (int i = 1; i < (NG > 0 ? NG : 1); ++i) res = res + term(i);
    } else {
      for (int i = 1; i < n; ++i) res = res + term(i);
    }
    return res;
  }
  double r0 = term(0), r1 = term(1), r2 = term(2), r3 = term(3), r4 = term(4), r5 = term(5), r6 = term(6),
         r7 = term(7);
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
    r0 = r0 + term(i); r1 = r1 + term(i + 1); r2 = r2 + term(i + 2); r3 = r3 + term(i + 3);
    r4 = r4 + term(i + 4); r5 = r5 + term(i + 5); r6 = r6 + term(i + 6); r7 = r7 + term(i + 7);
  }
  double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
  for (; i < n; ++i) res = res + term(i);
  return res;
}

// -------------------------------------------------------------- reductions
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum over the block; result valid in thread 0.  `scratch` holds >= 32 T.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  T r = (threadIdx.x < nw) ? scratch[threadIdx.x] : T(0);
  if (wid == 0) r = warp_sum(r);
  return r;
}

// hist[bin] += c for the lanes with `valid`; EVERY lane of the warp must call (converged).
// Values of one row crowd into a few histogram bins when the bins are cut from the top bits
// of a floating-point key (few binades in a row) or when most values are equal (wealth that
// underflowed to 0).  B200_HIST_ROUNDS rounds of "the lanes that share the first pending lane's
// bin add up (REDUX) and issue ONE atomic" take out the biggest crowds before the plain atomics.
// Default 0: measured in tally_select_kernel (clock stamps, C2's 45 561 tuples), the shared-memory
// atomic unit copes with the crowds better than the ballots / shuffles / REDUX of a round cost -
// pass 0 of the leverage with the most ties: 8.1k cycles plain, 6.7k with one round, 9.3k with
// two; of a leverage without: 4.2k / 6.8k / 9.2k.
#ifndef B200_HIST_ROUNDS
#define B200_HIST_ROUNDS 0
#endif
__device__ __forceinline__ void warp_hist_add(uint32_t* hist, uint32_t bin, uint32_t c, bool valid) {
  constexpr unsigned FULL = 0xffffffffu;
  if (B200_HIST_ROUNDS > 0) {
    unsigned rem = __ballot_sync(FULL, valid);
    const unsigned lane = threadIdx.x & 31;
#pragma unroll
    for (int round = 0; round < B200_HIST_ROUNDS; ++round) {
      if (rem == 0u) return;
      const int ld = __ffs(rem) - 1;
      const uint32_t lb = __shfl_sync(FULL, bin, ld);
      const bool same = valid && bin == lb;
      const unsigned grp = __ballot_sync(FULL, same);
      const uint32_t sum = __reduce_add_sync(FULL, same ? c : 0u);
      if (lane == (unsigned)ld && sum != 0u) atomicAdd(hist + lb, sum);
      rem &= ~grp;
      valid = valid && !same;
    }
  }
  if (valid && c != 0u) atomicAdd(hist + bin, c);
}

// Order-preserving map fp32 -> uint32 in torch.sort order (NaN greatest).
__host__ __device__ __forceinline__ uint32_t float_key(float f) {
  uint32_t b;
#ifdef __CUDA_ARCH__
  b = __float_as_uint(f);
#else
  union { float f; uint32_t u; } cv; cv.f = f; b = cv.u;
#endif
  if ((b & 0x7fffffffu) > 0x7f800000u) return 0xffffffffu;  // any NaN
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float key_float(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  if (k == 0xffffffffu) b = 0x7fc00000u;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  union { float f; uint32_t u; } cv; cv.u = b; return cv.f;
#endif
}

}  // namespace b200
