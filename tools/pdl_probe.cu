// Does programmatic dependent launch (PDL) survive what sits between two kernels in a stream?
// Build:  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o build/pdl_probe tools/pdl_probe.cu
//
// A primary kernel (one 128-thread block per SM) executes griddepcontrol.launch_dependents first and
// then spins for a fixed time; a secondary kernel, launched with the programmatic-stream-serialization
// attribute, stamps %globaltimer on entry, executes griddepcontrol.wait and stamps again.  Between the
// two launches the stream holds nothing, an event record (timing on / off), a wait on an event recorded
// earlier on the same stream, a wait on an event of another (idle) stream, or a wait on an event of another
// stream whose kernel runs longer than the primary.  One JSON line per case:
// overlap_us = last primary block's end - first secondary block's entry (> 0: the secondary started
// under the primary), wait_us = first secondary wait release - last primary end (the wait's latency),
// and for the last case after_other_us = first secondary entry - the other stream's kernel end (>= 0: the
// event wait held the secondary back although the primary had let it start).
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <vector>

#define CK(x)                                                                          \
  do {                                                                                 \
    cudaError_t e_ = (x);                                                              \
    if (e_ != cudaSuccess) {                                                           \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
      return 1;                                                                        \
    }                                                                                  \
  } while (0)

__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// stamps[2 * block] = entry, stamps[2 * block + 1] = end
__global__ void primary(unsigned long long* stamps, unsigned long long spin_ns) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const unsigned long long t0 = gtimer();
  while (gtimer() - t0 < spin_ns) {
  }
  __syncthreads();
  if (threadIdx.x == 0) { stamps[2 * blockIdx.x] = t0; stamps[2 * blockIdx.x + 1] = gtimer(); }
}

// stamps[2 * block] = entry (before the wait), stamps[2 * block + 1] = after the wait
__global__ void secondary(unsigned long long* stamps) {
  const unsigned long long t0 = gtimer();
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (threadIdx.x == 0) { stamps[2 * blockIdx.x] = t0; stamps[2 * blockIdx.x + 1] = gtimer(); }
}

int main() {
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  const unsigned long long spin_ns = 100000;   // 100 us
  unsigned long long *dp, *ds, *dq;
  CK(cudaMalloc(&dp, 2 * sms * sizeof(unsigned long long)));
  CK(cudaMalloc(&dq, 2 * sizeof(unsigned long long)));
  CK(cudaMalloc(&ds, 2 * sms * sizeof(unsigned long long)));
  cudaStream_t st, other;
  CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&other, cudaStreamNonBlocking));
  cudaEvent_t ev_plain, ev_timed, ev_same, ev_other;
  CK(cudaEventCreateWithFlags(&ev_plain, cudaEventDisableTiming));
  CK(cudaEventCreate(&ev_timed));
  CK(cudaEventCreateWithFlags(&ev_same, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&ev_other, cudaEventDisableTiming));
  const char* names[] = {"nothing", "event_record", "event_record_timing", "wait_same_stream_event",
                         "wait_other_stream_event", "no_pdl_attribute", "wait_other_stream_pending"};
  constexpr int NCASE = 7;
  std::vector<unsigned long long> hp(2 * sms), hs(2 * sms), hq(2);
  printf("{\"device\": \"%s\", \"sms\": %d, \"primary_spin_us\": %.1f}\n", prop.name, sms, spin_ns * 1e-3);
  for (int rep = 0; rep < 4; ++rep) {     // rep 0 warms up and is not printed
    for (int c = 0; c < NCASE; ++c) {
      CK(cudaEventRecord(ev_same, st));
      CK(cudaEventRecord(ev_other, other));
      CK(cudaStreamSynchronize(st));
      CK(cudaStreamSynchronize(other));
      if (c == 6) {   // one block for 3x the primary's time on the other stream, then the event
        primary<<<1, 32, 0, other>>>(dq, 3 * spin_ns);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ev_other, other));
      }
      primary<<<sms, 128, 0, st>>>(dp, spin_ns);
      CK(cudaGetLastError());
      if (c == 1) CK(cudaEventRecord(ev_plain, st));
      if (c == 2) CK(cudaEventRecord(ev_timed, st));
      if (c == 3) CK(cudaStreamWaitEvent(st, ev_same, 0));
      if (c == 4 || c == 6) CK(cudaStreamWaitEvent(st, ev_other, 0));
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(sms);
      cfg.blockDim = dim3(128);
      cfg.stream = st;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = at;
      cfg.numAttrs = c == 5 ? 0 : 1;
      CK(cudaLaunchKernelEx(&cfg, secondary, ds));
      CK(cudaStreamSynchronize(st));
      CK(cudaMemcpy(hp.data(), dp, hp.size() * 8, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(hs.data(), ds, hs.size() * 8, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(hq.data(), dq, hq.size() * 8, cudaMemcpyDeviceToHost));
      unsigned long long p_end = 0, s_start = ~0ull, s_wait = ~0ull;
      for (int b = 0; b < sms; ++b) {
        p_end = hp[2 * b + 1] > p_end ? hp[2 * b + 1] : p_end;
        s_start = hs[2 * b] < s_start ? hs[2 * b] : s_start;
        s_wait = hs[2 * b + 1] < s_wait ? hs[2 * b + 1] : s_wait;
      }
      if (rep > 0 && c == 6)
        printf("{\"case\": \"%s\", \"rep\": %d, \"overlap_us\": %.2f, \"after_other_us\": %.2f}\n", names[c], rep,
               ((double)p_end - (double)s_start) * 1e-3, ((double)s_start - (double)hq[1]) * 1e-3);
      else if (rep > 0)
        printf("{\"case\": \"%s\", \"rep\": %d, \"overlap_us\": %.2f, \"wait_us\": %.2f}\n", names[c], rep,
               ((double)p_end - (double)s_start) * 1e-3, ((double)s_wait - (double)p_end) * 1e-3);
    }
  }
  CK(cudaDeviceSynchronize());
  return 0;
}
