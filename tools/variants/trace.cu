// DEV ONLY (not part of the package): the shipped streaming shell with its timeline hooks turned on, for
// tools/prof_stream_timeline.py.  Thread 0 of every CTA takes a record slot at entry and writes %globaltimer at the
// five B200POSE_TRACE points of stream_kernel_tma (lie_kernels.cuh).
#include <stdint.h>
#include <cuda_runtime.h>

namespace b200trace {
constexpr unsigned kCap = 1u << 16;
// record: [0] first input pointer (identifies the launch), [1] blockIdx.x << 32 | smid, [2..6] time at points 0..4 (ns),
// [7] tiles of the CTA
__device__ unsigned g_count;
__device__ unsigned long long g_rec[kCap][8];
__device__ __forceinline__ unsigned long long now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ unsigned smid() {
  unsigned s;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(s));
  return s;
}
}  // namespace b200trace

#define B200POSE_TRACE(k) B200POSE_TRACE_##k
// point 0 sits at function scope: the slot it declares is visible to the later points
#define B200POSE_TRACE_0                                                                              \
  unsigned trace_slot_ = b200trace::kCap;                                                             \
  if (threadIdx.x == 0) {                                                                             \
    trace_slot_ = atomicAdd(&b200trace::g_count, 1u);                                                 \
    if (trace_slot_ < b200trace::kCap) {                                                              \
      b200trace::g_rec[trace_slot_][0] = (unsigned long long)(uintptr_t)p.in[0];                      \
      b200trace::g_rec[trace_slot_][1] = ((unsigned long long)blockIdx.x << 32) | b200trace::smid();   \
      b200trace::g_rec[trace_slot_][2] = b200trace::now();                                            \
    }                                                                                                 \
  }
#define B200POSE_TRACE_AT(k, extra)                                                                   \
  do {                                                                                                \
    if (threadIdx.x == 0 && trace_slot_ < b200trace::kCap) {                                          \
      b200trace::g_rec[trace_slot_][2 + k] = b200trace::now();                                        \
      extra;                                                                                          \
    }                                                                                                 \
  } while (0)
#define B200POSE_TRACE_1 B200POSE_TRACE_AT(1, (void)0)
#define B200POSE_TRACE_2 B200POSE_TRACE_AT(2, (void)0)
#define B200POSE_TRACE_3 B200POSE_TRACE_AT(3, (void)0)
#define B200POSE_TRACE_4 B200POSE_TRACE_AT(4, b200trace::g_rec[trace_slot_][7] = (unsigned long long)ntiles)

#include "lie_kernels.cuh"
using namespace b200pose;

#define TRACE_EXPORT extern "C" __attribute__((visibility("default")))
// the shipped entry points' launch path (launch_stream), instantiated with the hooks on
TRACE_EXPORT int trace_se3_exp_fwd_f32(const float* i0, float* o0, long long n, void* st) {
  const float* in[1] = {i0}; float* out[1] = {o0};
  return launch_stream<OpExpFwd<SE3g, float> >(in, out, n, (cudaStream_t)st);
}
TRACE_EXPORT int trace_SE3_log_fwd_f32(const float* i0, float* o0, long long n, void* st) {
  const float* in[1] = {i0}; float* out[1] = {o0};
  return launch_stream<OpLogFwd<SE3g, float> >(in, out, n, (cudaStream_t)st);
}
TRACE_EXPORT int trace_reset() {
  unsigned z = 0;
  return (int)cudaMemcpyToSymbol(b200trace::g_count, &z, sizeof(z));
}
// copies min(count, cap) records to host (8 u64 each); returns the number of slots taken (may exceed the cap)
TRACE_EXPORT long long trace_read(unsigned long long* host) {
  unsigned cnt = 0;
  if (cudaMemcpyFromSymbol(&cnt, b200trace::g_count, sizeof(cnt)) != cudaSuccess) return -1;
  unsigned m = cnt < b200trace::kCap ? cnt : b200trace::kCap;
  if (m && cudaMemcpyFromSymbol(host, b200trace::g_rec, (size_t)m * 64) != cudaSuccess) return -1;
  return cnt;
}
TRACE_EXPORT long long trace_capacity() { return b200trace::kCap; }

__global__ void timer_samples_kernel(unsigned long long* out, int n) {
  for (int i = 0; i < n; ++i) out[i] = b200trace::now();
}
// one thread reads %globaltimer n times back to back into dev_out (device buffer of n u64)
TRACE_EXPORT int trace_timer_samples(unsigned long long* dev_out, int n, void* st) {
  timer_samples_kernel<<<1, 1, 0, (cudaStream_t)st>>>(dev_out, n);
  return (int)cudaGetLastError();
}
