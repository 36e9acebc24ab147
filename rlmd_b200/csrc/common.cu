// Error plumbing and device queries shared by every entry point.
#include "common.cuh"

#include <cstdlib>
#include <cstring>

namespace b200 {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  return set_error(B200_ECUDA, "%s: %s", what, cudaGetErrorString(e));
}

bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("B200_PDL"); return e == nullptr || atoi(e) != 0; }();
  return on;
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return 148; }
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = 148;
    }
    cached[dev] = n;
  }
  return cached[dev];
}

// Multi-GPU statistics exchange: the integer and double words a phase must sum
// over ranks are gathered into ONE contiguous fp64 buffer (counts are far below
// 2^53, so their sums are exact in fp64), reduced by a single all-reduce - in the
// NVSwitch when NCCL uses NVLS - and scattered back.
__global__ void __launch_bounds__(256)
exchange_pack_kernel(const long long* __restrict__ ws, int64_t words, int64_t rows, int64_t io, int64_t ic,
                     int64_t d_o, int64_t dc, double* __restrict__ staging) {
  const int64_t per = ic + dc, total = rows * per;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / per, k = i - r * per;
    staging[i] = k < ic ? (double)ws[r * words + io + k] : __longlong_as_double(ws[r * words + d_o + (k - ic)]);
  }
}
__global__ void __launch_bounds__(256)
exchange_unpack_kernel(long long* __restrict__ ws, int64_t words, int64_t rows, int64_t io, int64_t ic, int64_t d_o,
                       int64_t dc, const double* __restrict__ staging) {
  const int64_t per = ic + dc, total = rows * per;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / per, k = i - r * per;
    if (k < ic) ws[r * words + io + k] = __double2ll_rn(staging[i]);
    else ws[r * words + d_o + (k - ic)] = __double_as_longlong(staging[i]);
  }
}

}  // namespace b200

extern "C" int b200_exchange_pack(const void* workspace, int64_t words_per_row, int64_t rows, int64_t int_offset,
                                  int64_t int_count, int64_t dbl_offset, int64_t dbl_count, double* staging,
                                  void* stream) {
  using namespace b200;
  B200_REQUIRE(rows >= 0 && int_count >= 0 && dbl_count >= 0, "exchange_pack: negative size");
  const int64_t total = rows * (int_count + dbl_count);
  if (total == 0) return 0;
  B200_REQUIRE(workspace && staging, "exchange_pack: NULL buffer");
  const int grid = (int)((total + 255) / 256 < (int64_t)sm_count() * 8 ? (total + 255) / 256 : (int64_t)sm_count() * 8);
  exchange_pack_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const long long*)workspace, words_per_row, rows,
                                                               int_offset, int_count, dbl_offset, dbl_count, staging);
  return check_cuda(cudaGetLastError(), "exchange_pack launch");
}

extern "C" int b200_exchange_unpack(void* workspace, int64_t words_per_row, int64_t rows, int64_t int_offset,
                                    int64_t int_count, int64_t dbl_offset, int64_t dbl_count, const double* staging,
                                    void* stream) {
  using namespace b200;
  B200_REQUIRE(rows >= 0 && int_count >= 0 && dbl_count >= 0, "exchange_unpack: negative size");
  const int64_t total = rows * (int_count + dbl_count);
  if (total == 0) return 0;
  B200_REQUIRE(workspace && staging, "exchange_unpack: NULL buffer");
  const int grid = (int)((total + 255) / 256 < (int64_t)sm_count() * 8 ? (total + 255) / 256 : (int64_t)sm_count() * 8);
  exchange_unpack_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((long long*)workspace, words_per_row, rows, int_offset,
                                                                 int_count, dbl_offset, dbl_count, staging);
  return check_cuda(cudaGetLastError(), "exchange_unpack launch");
}

extern "C" const char* b200_last_error(void) { return b200::g_err; }

extern "C" int b200_version(void) { return 100; }  // 0.1.0

extern "C" int b200_device_info(int32_t* sms, int32_t* cc_major, int32_t* cc_minor) {
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  int a = 0, b = 0, c = 0;
  B200_CUDA(cudaDeviceGetAttribute(&a, cudaDevAttrMultiProcessorCount, dev));
  B200_CUDA(cudaDeviceGetAttribute(&b, cudaDevAttrComputeCapabilityMajor, dev));
  B200_CUDA(cudaDeviceGetAttribute(&c, cudaDevAttrComputeCapabilityMinor, dev));
  if (sms) *sms = a;
  if (cc_major) *cc_major = b;
  if (cc_minor) *cc_minor = c;
  return 0;
}
