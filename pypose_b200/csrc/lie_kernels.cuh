// lie_kernels.cuh — HBM streaming shell + per-op functors for the LieTensor op family.
//
// Data layout in HBM: row-major (N, d) arrays with d in 3..9 words (12..72 B rows).  Rows are not
// 16-byte multiples, so a per-thread vector load would be misaligned; instead each CTA owns a
// contiguous chunk of elements and moves it tile-by-tile:
//
//   HBM --(16 B coalesced, streaming hint)--> smem tile --(row gather)--> registers
//        --(lie_math.cuh)--> registers --(row scatter)--> smem tile --(16 B coalesced)--> HBM
//
// so every DRAM sector is touched exactly once (algorithmic bytes == DRAM traffic).  The grid is a
// multiple of the SM count: each CTA gets the same number of elements (chunk), so there is no tail
// wave.  One element per thread per tile; EPT tiles are batched per barrier to raise bytes in flight.
#pragma once
#include "b200pose.h"   // every definition is checked against the generated declaration
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include "lie_ops.cuh"
#include "tma.cuh"

namespace b200pose {

constexpr int kThreads = 256;

template <typename T, int NIN, int NOUT> struct StreamParams {
  const T* in[NIN];
  T* out[NOUT];
  long long n;       // elements
  long long chunk;   // elements per CTA (multiple of 4)
  int vec_ok;        // all base pointers 16 B aligned
};

// cooperative copy of `nwords` T-words global -> shared (16 B vectors + scalar tail)
template <typename T>
__device__ __forceinline__ void tile_load(T* __restrict__ s, const T* __restrict__ g, int nwords, int vec_ok) {
  constexpr int WPV = 16 / sizeof(T);
  int nvec = vec_ok ? nwords / WPV : 0;
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4* s4 = reinterpret_cast<float4*>(s);
#pragma unroll 4
  for (int k = threadIdx.x; k < nvec; k += kThreads) s4[k] = __ldcs(g4 + k);
  for (int k = nvec * WPV + threadIdx.x; k < nwords; k += kThreads) s[k] = __ldcs(g + k);
}
template <typename T>
__device__ __forceinline__ void tile_store(T* __restrict__ g, const T* __restrict__ s, int nwords, int vec_ok) {
  constexpr int WPV = 16 / sizeof(T);
  int nvec = vec_ok ? nwords / WPV : 0;
  float4* g4 = reinterpret_cast<float4*>(g);
  const float4* s4 = reinterpret_cast<const float4*>(s);
#pragma unroll 4
  for (int k = threadIdx.x; k < nvec; k += kThreads) __stcs(g4 + k, s4[k]);
  for (int k = nvec * WPV + threadIdx.x; k < nwords; k += kThreads) __stcs(g + k, s[k]);
}

template <int D, typename T> __device__ __forceinline__ void row_get(const T* __restrict__ s, int row, T (&r)[D]) {
#pragma unroll
  for (int j = 0; j < D; ++j) r[j] = s[row * D + j];
}
template <int D, typename T> __device__ __forceinline__ void row_put(T* __restrict__ s, int row, const T (&r)[D]) {
#pragma unroll
  for (int j = 0; j < D; ++j) s[row * D + j] = r[j];
}

// Op interface:
//   using T; static constexpr int NIN, NOUT, DI0, DI1, DI2, DO0, DO1 (unused = 1);
//   static __device__ void apply(const T* i0, const T* i1, const T* i2, T* o0, T* o1);
template <class Op, int EPT>
__global__ void __launch_bounds__(kThreads) stream_kernel(StreamParams<typename Op::T, Op::NIN, Op::NOUT> p) {
  using T = typename Op::T;
  constexpr int TILE = kThreads * EPT;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  T* s_i0 = reinterpret_cast<T*>(smem_raw);
  T* s_i1 = s_i0 + TILE * Op::DI0;
  T* s_i2 = s_i1 + (Op::NIN > 1 ? TILE * Op::DI1 : 0);
  T* s_o0 = s_i2 + (Op::NIN > 2 ? TILE * Op::DI2 : 0);
  T* s_o1 = s_o0 + TILE * Op::DO0;

  long long begin = (long long)blockIdx.x * p.chunk;
  long long end = begin + p.chunk;
  if (end > p.n) end = p.n;

  for (long long base = begin; base < end; base += TILE) {
    int cnt = (end - base) < TILE ? (int)(end - base) : TILE;
    tile_load(s_i0, p.in[0] + base * Op::DI0, cnt * Op::DI0, p.vec_ok);
    if (Op::NIN > 1) tile_load(s_i1, p.in[Op::NIN > 1 ? 1 : 0] + base * Op::DI1, cnt * Op::DI1, p.vec_ok);
    if (Op::NIN > 2) tile_load(s_i2, p.in[Op::NIN > 2 ? 2 : 0] + base * Op::DI2, cnt * Op::DI2, p.vec_ok);
    __syncthreads();
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      int row = threadIdx.x + e * kThreads;
      if (row < cnt) {
        T i0[Op::DI0], i1[Op::DI1], i2[Op::DI2], o0[Op::DO0], o1[Op::DO1];
        row_get<Op::DI0>(s_i0, row, i0);
        if (Op::NIN > 1) row_get<Op::DI1>(s_i1, row, i1);
        if (Op::NIN > 2) row_get<Op::DI2>(s_i2, row, i2);
        Op::apply(i0, i1, i2, o0, o1);
        row_put<Op::DO0>(s_o0, row, o0);
        if (Op::NOUT > 1) row_put<Op::DO1>(s_o1, row, o1);
      }
    }
    __syncthreads();
    tile_store(p.out[0] + base * Op::DO0, s_o0, cnt * Op::DO0, p.vec_ok);
    if (Op::NOUT > 1) tile_store(p.out[Op::NOUT > 1 ? 1 : 0] + base * Op::DO1, s_o1, cnt * Op::DO1, p.vec_ok);
    // the next iteration's loads only touch s_i*, and its compute phase (which writes s_o*) is
    // separated from these stores by the __syncthreads after the loads.
  }
}

// ----------------------------------------------------------------------------
// v2 shell: persistent CTAs, 1-D TMA bulk copies (cp.async.bulk -> SASS UBLKCP) into a multi-stage
// shared-memory ring signalled by mbarriers, bulk stores back (cp.async.bulk.global.shared).
// One elected thread issues all copies, so the other threads spend their issue slots on math only
// and loads for tile i+S overlap the math of tile i *inside* a CTA (v1 relies on other CTAs for that,
// which fails when a single wave of CTAs runs in lock-step: ncu profiles/r1a).
// Requirements: all base pointers 16 B aligned and every tile a multiple of 4 elements (the launcher
// guarantees both; the <= 3 element remainder and unaligned tensors go through the v1 kernel).
// ----------------------------------------------------------------------------
template <class Op, int S, int OS, int THREADS = kThreads, int EPT = 1> struct TmaLayout {
  using T = typename Op::T;
  static constexpr int TILE = THREADS * EPT;
  static constexpr int IN_WORDS = TILE * (Op::DI0 + (Op::NIN > 1 ? Op::DI1 : 0) + (Op::NIN > 2 ? Op::DI2 : 0));
  static constexpr int OUT_WORDS = TILE * (Op::DO0 + (Op::NOUT > 1 ? Op::DO1 : 0));
  static constexpr int BYTES = (S * IN_WORDS + OS * OUT_WORDS) * (int)sizeof(T) + 8 * S;
};

// Timeline probe hooks (tools/variants/trace.cu defines them; the shipped library expands them to nothing).
// B200POSE_TRACE(k) runs in stream_kernel_tma at k = 0 entry, 1 after griddepcontrol.wait, 2 tile 0 landed,
// 3 last store issued (thread 0), 4 exit.
#ifndef B200POSE_TRACE
#define B200POSE_TRACE(k)
#endif

// THREADS threads per CTA, EPT rows per thread per tile (rows tid, tid + THREADS, ...), S input / OS output stages.
// PF: tiles of the CTA's inputs hinted into L2 before the dependency wait (0 = none).
template <class Op, int S, int OS, int THREADS = kThreads, int EPT = 1, int PF = S>
__global__ void __launch_bounds__(THREADS) stream_kernel_tma(StreamParams<typename Op::T, Op::NIN, Op::NOUT> p) {
  using T = typename Op::T;
  using L = TmaLayout<Op, S, OS, THREADS, EPT>;
  constexpr int TILE = L::TILE;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  T* s_in = reinterpret_cast<T*>(smem_raw);
  T* s_out = s_in + S * L::IN_WORDS;
  uint64_t* full = reinterpret_cast<uint64_t*>(s_out + OS * L::OUT_WORDS);

  const long long begin = (long long)blockIdx.x * p.chunk;
  long long end = begin + p.chunk;
  if (end > p.n) end = p.n;
  const int ntiles = begin < end ? (int)((end - begin + TILE - 1) / TILE) : 0;
  const int tid = threadIdx.x;

  B200POSE_TRACE(0);
  // Programmatic dependent launch: let the next kernel in the stream start its launch/prologue now (its CTAs take
  // the SM slots this grid leaves free), and hold our own first load until the previous kernel has completed and
  // flushed.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // Warm L2 with the first PF tiles of every input while the previous grid drains.  Safe before the wait: a
    // prefetch is only a hint, never the value a load returns; L2 is the device's point of coherence, and every
    // load below is issued after griddepcontrol.wait, so it sees all writes of the previous grid (the Exp -> Log
    // chain reads what the previous launch wrote).  [begin, pf_end) lies within [0, n) and both ends are multiples
    // of 4 rows, so addresses and sizes are 16-byte multiples like the bulk loads'.  At most PF tiles per CTA:
    // bounded by the grid's ring footprint, so a large batch cannot flush L2 with hints.
    if (PF > 0 && begin < end) {
      const long long pf_end = end - begin > (long long)PF * TILE ? begin + (long long)PF * TILE : end;
      const uint32_t rows = (uint32_t)(pf_end - begin);
      bulk_prefetch_l2(p.in[0] + begin * Op::DI0, rows * Op::DI0 * sizeof(T));
      if (Op::NIN > 1) bulk_prefetch_l2(p.in[Op::NIN > 1 ? 1 : 0] + begin * Op::DI1, rows * Op::DI1 * sizeof(T));
      if (Op::NIN > 2) bulk_prefetch_l2(p.in[Op::NIN > 2 ? 2 : 0] + begin * Op::DI2, rows * Op::DI2 * sizeof(T));
    }
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  B200POSE_TRACE(1);
  __syncthreads();

  const int last_cnt = ntiles ? (int)(end - begin - (long long)(ntiles - 1) * TILE) : 0;

  auto issue_load = [&](int t, int s) {   // thread 0 only: tile t -> stage s
    const long long base = begin + (long long)t * TILE;
    const int cnt = (t == ntiles - 1) ? last_cnt : TILE;
    T* dst = s_in + s * L::IN_WORDS;
    const uint32_t b0 = cnt * Op::DI0 * sizeof(T), b1 = Op::NIN > 1 ? cnt * Op::DI1 * sizeof(T) : 0,
                   b2 = Op::NIN > 2 ? cnt * Op::DI2 * sizeof(T) : 0;
    mbar_expect_tx(&full[s], b0 + b1 + b2);
    bulk_g2s(dst, p.in[0] + base * Op::DI0, b0, &full[s]);
    if (Op::NIN > 1) bulk_g2s(dst + TILE * Op::DI0, p.in[Op::NIN > 1 ? 1 : 0] + base * Op::DI1, b1, &full[s]);
    if (Op::NIN > 2)
      bulk_g2s(dst + TILE * (Op::DI0 + Op::DI1), p.in[Op::NIN > 2 ? 2 : 0] + base * Op::DI2, b2, &full[s]);
  };

  if (tid == 0) {
    const int pre = ntiles < S ? ntiles : S;
    for (int t = 0; t < pre; ++t) issue_load(t, t);
  }

  int s = 0, os = 0;          // running stage indices (no i % S in the loop)
  uint32_t parity = 0;
  for (int i = 0; i < ntiles; ++i) {
    const int cnt = (i == ntiles - 1) ? last_cnt : TILE;
    const T* in0 = s_in + s * L::IN_WORDS;
    const T* in1 = in0 + TILE * Op::DI0;
    const T* in2 = in1 + (Op::NIN > 1 ? TILE * Op::DI1 : 0);
    T* out0 = s_out + os * L::OUT_WORDS;
    T* out1 = out0 + TILE * Op::DO0;

    mbar_wait(&full[s], parity);
    if (i == 0) B200POSE_TRACE(2);
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int row = tid + e * THREADS;
      if (row < cnt) {
        T i0[Op::DI0], i1[Op::DI1], i2[Op::DI2], o0[Op::DO0], o1[Op::DO1];
        row_get<Op::DI0>(in0, row, i0);
        if (Op::NIN > 1) row_get<Op::DI1>(in1, row, i1);
        if (Op::NIN > 2) row_get<Op::DI2>(in2, row, i2);
        Op::apply(i0, i1, i2, o0, o1);
        row_put<Op::DO0>(out0, row, o0);
        if (Op::NOUT > 1) row_put<Op::DO1>(out1, row, o1);
      }
    }
    // out[(i+1) % OS] is written next iteration: its previous store (tile i+1-OS) must have been read
    // out of shared memory.  Stores pending now: tiles <= i-1; allow the newest OS-2 of them to stay.
    if (tid == 0) bulk_wait_read<(OS >= 2 ? OS - 2 : 0)>();
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      const long long base = begin + (long long)i * TILE;
      bulk_s2g(p.out[0] + base * Op::DO0, out0, cnt * Op::DO0 * sizeof(T));
      if (Op::NOUT > 1) bulk_s2g(p.out[Op::NOUT > 1 ? 1 : 0] + base * Op::DO1, out1, cnt * Op::DO1 * sizeof(T));
      bulk_commit();
      if (i + S < ntiles) issue_load(i + S, s);
      if (i == ntiles - 1) B200POSE_TRACE(3);
    }
    if (++s == S) { s = 0; parity ^= 1; }
    if (++os == OS) os = 0;
  }
  // Only the shared-memory reads of the stores must finish before the CTA frees its slot; their global writes are
  // covered by grid completion, which is what the next kernel's griddepcontrol.wait (or stream order) waits for.
  if (tid == 0) bulk_wait_read<0>();
  B200POSE_TRACE(4);
}

constexpr int kMaxDevices = 64;
inline int current_device_slot() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev >= 0 && dev < kMaxDevices ? dev : 0;
}
struct DeviceInfo { int sms; };
inline const DeviceInfo& device_info() {
  static thread_local int cached_dev = -1;
  static thread_local DeviceInfo info;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev != cached_dev) {
    cudaDeviceGetAttribute(&info.sms, cudaDevAttrMultiProcessorCount, dev);
    cached_dev = dev;
  }
  return info;
}

template <class Op, int EPT>
int launch_stream_ept(const typename Op::T* const* in, typename Op::T* const* out, long long n, cudaStream_t stream) {
  using T = typename Op::T;
  constexpr int TILE = kThreads * EPT;
  constexpr int words = TILE * (Op::DI0 + (Op::NIN > 1 ? Op::DI1 : 0) + (Op::NIN > 2 ? Op::DI2 : 0) + Op::DO0 +
                                (Op::NOUT > 1 ? Op::DO1 : 0));
  constexpr int smem = words * (int)sizeof(T);
  auto kern = stream_kernel<Op, EPT>;
  // the dynamic-smem attribute is per device: cache the occupancy per (kernel instantiation, device)
  static thread_local int occ_dev[kMaxDevices] = {};
  int& occ = occ_dev[current_device_slot()];
  if (occ == 0) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kThreads, smem);
    if (occ < 1) occ = 1;
  }
  StreamParams<T, Op::NIN, Op::NOUT> p;
  uintptr_t align = 0;
  for (int i = 0; i < Op::NIN; ++i) { p.in[i] = in[i]; align |= reinterpret_cast<uintptr_t>(in[i]); }
  for (int i = 0; i < Op::NOUT; ++i) { p.out[i] = out[i]; align |= reinterpret_cast<uintptr_t>(out[i]); }
  p.vec_ok = (align & 15) == 0;
  p.n = n;
  long long tiles = (n + TILE - 1) / TILE;
  long long slots = (long long)device_info().sms * occ;
  long long grid = tiles < slots ? tiles : slots;
  long long chunk = (n + grid - 1) / grid;
  chunk = (chunk + 3) & ~3LL;
  grid = (n + chunk - 1) / chunk;
  p.chunk = chunk;
  kern<<<(unsigned)grid, kThreads, smem, stream>>>(p);
  return (int)cudaGetLastError();
}

// B200POSE_STREAM=v1 forces the plain-load shell (A/B measurements); B200POSE_CTAS_PER_SM caps residency.
inline int stream_impl_v1() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("B200POSE_STREAM"); v = (e && e[0] == 'v' && e[1] == '1') ? 1 : 0; }
  return v;
}
inline int stream_pdl() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("B200POSE_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
  return v;
}
inline int stream_max_ctas_per_sm() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("B200POSE_CTAS_PER_SM"); v = e ? atoi(e) : 8; if (v < 1) v = 8; }
  return v;
}

template <class Op, int S, int OS, int THREADS = kThreads, int EPT = 1, int PF = S>
int launch_stream_tma(const typename Op::T* const* in, typename Op::T* const* out, long long n, cudaStream_t stream) {
  using T = typename Op::T;
  using L = TmaLayout<Op, S, OS, THREADS, EPT>;
  auto kern = stream_kernel_tma<Op, S, OS, THREADS, EPT, PF>;
  static thread_local int occ_dev[kMaxDevices] = {};
  int& occ = occ_dev[current_device_slot()];
  if (occ == 0) {
    if (L::BYTES > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::BYTES);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, THREADS, L::BYTES);
    if (occ < 1) occ = 1;
    if (occ > stream_max_ctas_per_sm()) occ = stream_max_ctas_per_sm();
  }
  StreamParams<T, Op::NIN, Op::NOUT> p;
  for (int i = 0; i < Op::NIN; ++i) p.in[i] = in[i];
  for (int i = 0; i < Op::NOUT; ++i) p.out[i] = out[i];
  p.vec_ok = 1;
  p.n = n;
  long long tiles = (n + L::TILE - 1) / L::TILE;
  // With PDL, a shell whose SM holds >= 6 CTAs takes half of them per launch, so the next launch's CTAs are resident
  // (and warm L2 with their first tiles) while this one drains, instead of each boundary waiting for the whole grid
  // to exit.  With fewer slots (fp64, multi-operand rows) half a machine keeps too few bytes in flight: full grid.
  const int per_sm = stream_pdl() && occ >= 6 ? occ / 2 : occ;
  long long slots = (long long)device_info().sms * per_sm;
  long long grid = tiles < slots ? tiles : slots;
  long long chunk = (n + grid - 1) / grid;
  chunk = (chunk + 3) & ~3LL;
  grid = (n + chunk - 1) / chunk;
  p.chunk = chunk;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = L::BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = stream_pdl() ? 1 : 0;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, p);
  return e != cudaSuccess ? (int)e : (int)cudaGetLastError();
}

template <class Op>
int launch_stream_v1(const typename Op::T* const* in, typename Op::T* const* out, long long n, cudaStream_t stream) {
  // two rows per thread per barrier once there is enough work to fill the machine twice over
  if (n >= 2LL * kThreads * 2 * device_info().sms * 4 && sizeof(typename Op::T) == 4)
    return launch_stream_ept<Op, 2>(in, out, n, stream);
  return launch_stream_ept<Op, 1>(in, out, n, stream);
}

template <class Op>
int launch_stream(const typename Op::T* const* in, typename Op::T* const* out, long long n, cudaStream_t stream) {
  using T = typename Op::T;
  if (n <= 0) return 0;
  uintptr_t align = 0;
  for (int i = 0; i < Op::NIN; ++i) align |= reinterpret_cast<uintptr_t>(in[i]);
  for (int i = 0; i < Op::NOUT; ++i) align |= reinterpret_cast<uintptr_t>(out[i]);
  const long long n4 = n & ~3LL;
  if ((align & 15) != 0 || n4 == 0 || stream_impl_v1()) return launch_stream_v1<Op>(in, out, n, stream);
  constexpr int S = sizeof(T) == 4 ? 3 : 2;
  constexpr int OS = 2;
  int rc = launch_stream_tma<Op, S, OS>(in, out, n4, stream);
  if (rc != 0 || n4 == n) return rc;
  // <= 3 trailing elements: plain-load kernel on offset pointers
  const T* in_t[3] = {nullptr, nullptr, nullptr};
  T* out_t[2] = {nullptr, nullptr};
  const int di[3] = {Op::DI0, Op::DI1, Op::DI2};
  const int dout[2] = {Op::DO0, Op::DO1};
  for (int i = 0; i < Op::NIN; ++i) in_t[i] = in[i] + n4 * di[i];
  for (int i = 0; i < Op::NOUT; ++i) out_t[i] = out[i] + n4 * dout[i];
  return launch_stream_ept<Op, 1>(in_t, out_t, n - n4, stream);
}

// ----------------------------------------------------------------------------
// C-ABI launchers
// ----------------------------------------------------------------------------
#define B200_EXPORT extern "C" __attribute__((visibility("default")))

#define ABI_1_1(NAME, OPT, G, CT)                                                              \
  B200_EXPORT int NAME(const CT* i0, CT* o0, long long n, void* stream) {                  \
    const CT* in[1] = {i0}; CT* out[1] = {o0};                                             \
    return launch_stream<OPT<G, CT> >(in, out, n, (cudaStream_t)stream);                            \
  }
#define ABI_2_1(NAME, OPT, G, CT)                                                              \
  B200_EXPORT int NAME(const CT* i0, const CT* i1, CT* o0, long long n, void* stream) {    \
    const CT* in[2] = {i0, i1}; CT* out[1] = {o0};                                         \
    return launch_stream<OPT<G, CT> >(in, out, n, (cudaStream_t)stream);                            \
  }
#define ABI_2_2(NAME, OPT, G, CT)                                                              \
  B200_EXPORT int NAME(const CT* i0, const CT* i1, CT* o0, CT* o1, long long n, void* stream) { \
    const CT* in[2] = {i0, i1}; CT* out[2] = {o0, o1};                                     \
    return launch_stream<OPT<G, CT> >(in, out, n, (cudaStream_t)stream);                            \
  }
#define ABI_3_2(NAME, OPT, G, CT)                                                              \
  B200_EXPORT int NAME(const CT* i0, const CT* i1, const CT* i2, CT* o0, CT* o1, long long n, void* stream) { \
    const CT* in[3] = {i0, i1, i2}; CT* out[2] = {o0, o1};                                 \
    return launch_stream<OPT<G, CT> >(in, out, n, (cudaStream_t)stream);                            \
  }

// one group x one dtype: 17 entry points.  alg = lower-case algebra name, GRP = group name.
#define B200_GROUP_OPS(alg, GRP, G, CT, SFX)                                               \
  ABI_1_1(b200_##alg##_exp_fwd_##SFX, OpExpFwd, G, CT)                               \
  ABI_2_1(b200_##alg##_exp_bwd_##SFX, OpExpBwd, G, CT)                               \
  ABI_1_1(b200_##GRP##_log_fwd_##SFX, OpLogFwd, G, CT)                               \
  ABI_2_1(b200_##GRP##_log_bwd_##SFX, OpLogBwd, G, CT)                               \
  ABI_1_1(b200_##GRP##_inv_fwd_##SFX, OpInvFwd, G, CT)                               \
  ABI_2_1(b200_##GRP##_inv_bwd_##SFX, OpInvBwd, G, CT)                               \
  ABI_2_1(b200_##GRP##_mul_fwd_##SFX, OpMulFwd, G, CT)                               \
  ABI_2_2(b200_##GRP##_mul_bwd_##SFX, OpMulBwd, G, CT)                               \
  ABI_2_1(b200_##GRP##_act_fwd_##SFX, OpActFwd, G, CT)                               \
  ABI_3_2(b200_##GRP##_act_bwd_##SFX, OpActBwd, G, CT)                               \
  ABI_2_1(b200_##GRP##_act4_fwd_##SFX, OpAct4Fwd, G, CT)                             \
  ABI_3_2(b200_##GRP##_act4_bwd_##SFX, OpAct4Bwd, G, CT)                             \
  ABI_2_1(b200_##GRP##_adj_fwd_##SFX, OpAdjFwd, G, CT)                               \
  ABI_3_2(b200_##GRP##_adj_bwd_##SFX, OpAdjBwd, G, CT)                               \
  ABI_2_1(b200_##GRP##_adjt_fwd_##SFX, OpAdjTFwd, G, CT)                             \
  ABI_3_2(b200_##GRP##_adjt_bwd_##SFX, OpAdjTBwd, G, CT)                             \
  ABI_2_1(b200_##GRP##_jinvp_fwd_##SFX, OpJinvpFwd, G, CT)

}  // namespace b200pose
