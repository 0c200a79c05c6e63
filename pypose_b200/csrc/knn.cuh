// knn.cuh — brute-force k-nearest-neighbour search (pp.knn) and the fused ICP correspondence step (pp.module.ICP).
//
// Reference: pypose/function/geometry.py:228-313 (`knn`: builds the full (..., N1, N2, D) difference tensor, takes its
// norm and calls topk) and pypose/module/icp.py (knn + gather + svdtf per iteration).
//
// One thread owns Q queries (Q = 4, 2, 1 for K <= 8, 16, 32) held in registers together with a sorted top-K list per
// query.  The CTA walks the neighbour cloud in tiles of TILE points, staged into shared memory by cp.async with double
// buffering; every thread reads each staged point once (a broadcast load) and tests it against its Q queries, so a
// shared load feeds Q distance evaluations.  A candidate is first compared with the current K-th key and only then
// inserted (branch-free shift through the list).  Selection for ord 2 works on squared distances; the square root is
// taken once, at output.
//
// Keys are the IEEE bit patterns of the (non-negative) distances, reinterpreted as unsigned integers: their order is
// the order of the distances, and a NaN sorts above +inf, as torch.topk orders it.  largest=True flips the magnitude
// bits, which reverses the order (NaN first).  The scan visits neighbours in increasing index order and never lets an
// equal key overtake, so ties keep the lower neighbour index.
//
// When B * ceil(N1 / (128 Q)) CTAs cannot fill the GPU, the neighbour range is split over `splits` CTAs per query
// block.  Each writes its partial top-K list to a workspace and a merge kernel combines them in split order, which
// keeps the tie rule.  The split is chosen from the shapes by b200_knn_plan.
//
// The ICP step (D = 3, K = 1) transforms each source point by the current SE3 estimate on the fly, finds its nearest
// target point and accumulates per-batch fp64 moments [count, sum s', sum t, sum t s'^T (row-major), sum distance]:
// the centred cross-covariance is formed from raw moments on the host side, which fp32 would cancel for clouds far
// from the origin.  The per-CTA sums are added with fp64 atomics, so their order (and the last bits) can vary.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <algorithm>
#include "lie_math.cuh"
#include "tma.cuh"

namespace b200pose {
namespace knn {

constexpr int THREADS = 128;
constexpr int TILE = 256;            // neighbour points per shared-memory stage
constexpr int NMOM = 17;             // ICP moments per batch

template <typename T> struct Key;
template <> struct Key<float> {
  using U = uint32_t;
  static constexpr U MAG = 0x7fffffffu;
  static __device__ __forceinline__ U bits(float x) { return __float_as_uint(x); }
  static __device__ __forceinline__ float value(U u) { return __uint_as_float(u); }
};
template <> struct Key<double> {
  using U = unsigned long long;
  static constexpr U MAG = 0x7fffffffffffffffull;
  static __device__ __forceinline__ U bits(double x) { return (U)__double_as_longlong(x); }
  static __device__ __forceinline__ double value(U u) { return __longlong_as_double((long long)u); }
};

template <int K> constexpr int queries_per_thread() { return K >= 32 ? 1 : K >= 16 ? 2 : 4; }

// max that propagates NaN, as torch.linalg.vector_norm(ord=inf) does
__device__ __forceinline__ float max_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ double max_nan(double a, double b) { return (b > a || b != b) ? b : a; }

// ord 2: squared distance; ord 1: sum |e|; ord 0 (inf): max |e|
template <typename T, int D, int ORD>
__device__ __forceinline__ T dist(const T* q, const T* p) {
  T acc = T(0);
#pragma unroll
  for (int d = 0; d < D; ++d) {
    const T e = q[d] - p[d];
    if (ORD == 2) acc = fma(e, e, acc);
    else if (ORD == 1) acc += fabs(e);
    else acc = max_nan(acc, fabs(e));
  }
  return acc;
}

template <typename T, int ORD>
__device__ __forceinline__ T finish(typename Key<T>::U key, typename Key<T>::U flip) {
  const T d = Key<T>::value(key ^ flip);
  return ORD == 2 ? sqrt(d) : d;
}

// sorted ascending list of the K smallest keys seen; an equal key never overtakes one already listed
template <typename U, int K>
struct TopK {
  U key[K];
  int idx[K];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int r = 0; r < K; ++r) { key[r] = ~U(0); idx[r] = -1; }
  }
  __device__ __forceinline__ void insert(U c, int j) {
#pragma unroll
    for (int i = K - 1; i > 0; --i) {
      const bool shift = key[i - 1] > c;
      idx[i] = shift ? idx[i - 1] : (key[i] > c ? j : idx[i]);
      key[i] = shift ? key[i - 1] : (key[i] > c ? c : key[i]);
    }
    idx[0] = key[0] > c ? j : idx[0];
    key[0] = key[0] > c ? c : key[0];
  }
  __device__ __forceinline__ void push(U c, int j) {
    if (c < key[K - 1]) insert(c, j);
  }
};

template <typename T>
struct Args {
  const T* ref;  const T* nbr;
  long long ref_bs, nbr_bs;            // elements between batches, 0 = one cloud for every batch
  long long N1, N2, chunk;             // chunk: neighbours per split (multiple of TILE)
  int qblocks, S, k;
  typename Key<T>::U flip;             // 0, or Key<T>::MAG for largest=True
  T* vals;  long long* inds;           // (B, N1, k) outputs when S == 1
  typename Key<T>::U* wkey;  int* widx;// (B, N1, S, K) partial lists when S > 1
  const T* pose;  double* mom;         // ICP: (B, 7) current SE3, (B, NMOM) moments
};

__device__ __forceinline__ void cp_async(float* s, const float* g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(s)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async(double* s, const double* g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(s)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <typename T>
__device__ __forceinline__ void stage(T* dst, const T* src, int n) {
  for (int e = threadIdx.x; e < n; e += THREADS) cp_async(dst + e, src + e);
  cp_commit();
}

template <typename T>
__device__ __forceinline__ V3<T> icp_transform(const T* pose, const T* p) {
  Q4<T> q = ldq(pose + 3);
  return qrot(q, ld3(p)) + ld3(pose);
}

// per-query moments of one ICP correspondence, summed over the CTA and added to mom[0..NMOM)
template <typename T>
__device__ __forceinline__ void add_moment(double* m, const V3<T>& s, const T* t, T d) {
  const double sv[3] = {(double)s.x, (double)s.y, (double)s.z};
  m[0] += 1.0;
#pragma unroll
  for (int a = 0; a < 3; ++a) { m[1 + a] += sv[a]; m[4 + a] += (double)t[a]; }
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int c = 0; c < 3; ++c) m[7 + 3 * a + c] += (double)t[a] * sv[c];
  m[16] += (double)d;
}

__device__ __forceinline__ void reduce_moments(double* m, double* mom, void* smem) {
  double* red = reinterpret_cast<double*>(smem);   // (THREADS / 32, NMOM)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int r = 0; r < NMOM; ++r) {
    double v = m[r];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp * NMOM + r] = v;
  }
  __syncthreads();
  if (threadIdx.x < NMOM) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) v += red[w * NMOM + threadIdx.x];
    atomicAdd(mom + threadIdx.x, v);
  }
}

// grid (B * qblocks, S).  ICP implies D == 3 and K == 1.
template <typename T, int D, int ORD, int K, bool ICP>
__global__ void __launch_bounds__(THREADS, 1) knn_kernel(const Args<T> a) {
  using U = typename Key<T>::U;
  constexpr int Q = queries_per_thread<K>();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* tiles = reinterpret_cast<T*>(smem_raw);       // (2, TILE, D)
  const long long b = blockIdx.x / a.qblocks;
  const int qb = blockIdx.x % a.qblocks, s = blockIdx.y;
  const T* ref = a.ref + b * a.ref_bs;
  const T* nbr = a.nbr + b * a.nbr_bs;

  T q[Q][D];
  TopK<U, K> top[Q];
  const long long i0 = (long long)qb * THREADS * Q + threadIdx.x;
#pragma unroll
  for (int u = 0; u < Q; ++u) {
    const long long i = i0 + (long long)u * THREADS;
    if constexpr (ICP) {
      const T zero[3] = {T(0), T(0), T(0)};
      const V3<T> p = icp_transform(a.pose + b * 7, i < a.N1 ? ref + i * 3 : zero);
      q[u][0] = p.x; q[u][1] = p.y; q[u][2] = p.z;
    } else {
#pragma unroll
      for (int d = 0; d < D; ++d) q[u][d] = i < a.N1 ? ref[i * D + d] : T(0);
    }
    top[u].init();
  }

  const long long j0 = (long long)s * a.chunk;
  const long long j1 = min(a.N2, j0 + a.chunk);
  const int ntiles = (int)((j1 - j0 + TILE - 1) / TILE);
  stage(tiles, nbr + j0 * D, (int)min((long long)TILE, j1 - j0) * D);
  for (int t = 0; t < ntiles; ++t) {
    const long long jb = j0 + (long long)t * TILE;
    const int n = (int)min((long long)TILE, j1 - jb);
    if (t + 1 < ntiles) {
      stage(tiles + ((t + 1) & 1) * TILE * D, nbr + (jb + TILE) * D, (int)min((long long)TILE, j1 - jb - TILE) * D);
      cp_wait<1>();
    } else {
      cp_wait<0>();
    }
    __syncthreads();
    const T* p = tiles + (t & 1) * TILE * D;
    auto visit = [&](int jj) {
      T pt[D];
#pragma unroll
      for (int d = 0; d < D; ++d) pt[d] = p[jj * D + d];
#pragma unroll
      for (int u = 0; u < Q; ++u) top[u].push(Key<T>::bits(dist<T, D, ORD>(q[u], pt)) ^ a.flip, (int)jb + jj);
    };
    if (n == TILE) {
#pragma unroll 4
      for (int jj = 0; jj < TILE; ++jj) visit(jj);
    } else {
      for (int jj = 0; jj < n; ++jj) visit(jj);
    }
    __syncthreads();
  }

  if (a.S > 1) {
#pragma unroll
    for (int u = 0; u < Q; ++u) {
      const long long i = i0 + (long long)u * THREADS;
      if (i >= a.N1) continue;
      const long long o = ((b * a.N1 + i) * a.S + s) * K;
#pragma unroll
      for (int r = 0; r < K; ++r) { a.wkey[o + r] = top[u].key[r]; a.widx[o + r] = top[u].idx[r]; }
    }
    return;
  }
  if constexpr (ICP) {
    double m[NMOM];
#pragma unroll
    for (int r = 0; r < NMOM; ++r) m[r] = 0.0;
#pragma unroll
    for (int u = 0; u < Q; ++u) {
      const long long i = i0 + (long long)u * THREADS;
      if (i < a.N1)
        add_moment(m, mk(q[u][0], q[u][1], q[u][2]), nbr + (long long)top[u].idx[0] * 3,
                   finish<T, ORD>(top[u].key[0], a.flip));
    }
    reduce_moments(m, a.mom + b * NMOM, smem_raw);   // the last __syncthreads of the tile loop freed the tiles
  } else {
#pragma unroll
    for (int u = 0; u < Q; ++u) {
      const long long i = i0 + (long long)u * THREADS;
      if (i >= a.N1) continue;
      const long long o = (b * a.N1 + i) * a.k;
#pragma unroll
      for (int r = 0; r < K; ++r)
        if (r < a.k) { a.vals[o + r] = finish<T, ORD>(top[u].key[r], a.flip); a.inds[o + r] = top[u].idx[r]; }
    }
  }
}

// grid (ceil(N1 / THREADS), B): one thread per query merges its S partial lists in split order
template <typename T, int ORD, int K, bool ICP>
__global__ void __launch_bounds__(THREADS, 1) merge_kernel(const Args<T> a) {
  using U = typename Key<T>::U;
  __shared__ double red[(THREADS / 32) * NMOM];
  const long long b = blockIdx.y;
  const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
  TopK<U, K> top;
  top.init();
  if (i < a.N1) {
    const long long o = (b * a.N1 + i) * a.S * K;
    for (int s = 0; s < a.S; ++s)
#pragma unroll
      for (int r = 0; r < K; ++r) top.push(a.wkey[o + s * K + r], a.widx[o + s * K + r]);
  }
  if constexpr (ICP) {
    double m[NMOM];
#pragma unroll
    for (int r = 0; r < NMOM; ++r) m[r] = 0.0;
    if (i < a.N1)
      add_moment(m, icp_transform(a.pose + b * 7, a.ref + b * a.ref_bs + i * 3),
                 a.nbr + b * a.nbr_bs + (long long)top.idx[0] * 3, finish<T, ORD>(top.key[0], a.flip));
    reduce_moments(m, a.mom + b * NMOM, red);
  } else if (i < a.N1) {
    const long long o = (b * a.N1 + i) * a.k;
#pragma unroll
    for (int r = 0; r < K; ++r)
      if (r < a.k) { a.vals[o + r] = finish<T, ORD>(top.key[r], a.flip); a.inds[o + r] = top.idx[r]; }
  }
}

inline int round_k(int k) { int K = 1; while (K < k) K <<= 1; return K; }
inline int qpt(int K) { return K >= 32 ? 1 : K >= 16 ? 2 : 4; }
inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

// Split rule: keep at least 4 CTAs per SM.  Each split covers whole tiles, at least one, and the partial lists
// stay within 32 MB.  Returns the workspace bytes; *splits receives S (1 = no split, no workspace).
inline long long plan(long long B, long long N1, long long N2, int k, int elem_size, int sms, long long* splits) {
  const int K = round_k(k);
  const long long ctas = B * cdiv(N1, (long long)THREADS * qpt(K));
  const long long per = (long long)K * (elem_size + 4);
  long long S = 1;
  if (ctas > 0 && ctas < 4LL * sms) {
    S = cdiv(4LL * sms, ctas);
    S = std::min(S, std::max(1LL, N2 / TILE));
    S = std::min(S, std::max(1LL, (32LL << 20) / std::max(1LL, B * N1 * per)));
    S = std::min(S, 1024LL);
  }
  if (S > 1) S = cdiv(N2, cdiv(cdiv(N2, S), TILE) * TILE);   // no empty split
  *splits = S;
  return S > 1 ? B * N1 * S * per : 0;
}

template <typename T, int D, int ORD, int K, bool ICP>
int launch(Args<T> a, long long B, cudaStream_t st) {
  a.qblocks = (int)cdiv(a.N1, (long long)THREADS * queries_per_thread<K>());
  a.chunk = a.S > 1 ? cdiv(cdiv(a.N2, a.S), TILE) * TILE : a.N2;
  const size_t smem = 2 * TILE * D * sizeof(T);
  knn_kernel<T, D, ORD, K, ICP><<<dim3((unsigned)(B * a.qblocks), (unsigned)a.S), THREADS, smem, st>>>(a);
  if (a.S > 1) merge_kernel<T, ORD, K, ICP><<<dim3((unsigned)cdiv(a.N1, THREADS), (unsigned)B), THREADS, 0, st>>>(a);
  return (int)cudaGetLastError();
}

template <typename T, int D, int ORD>
int by_k(Args<T> a, long long B, cudaStream_t st) {
  switch (round_k(a.k)) {
    case 1: return launch<T, D, ORD, 1, false>(a, B, st);
    case 2: return launch<T, D, ORD, 2, false>(a, B, st);
    case 4: return launch<T, D, ORD, 4, false>(a, B, st);
    case 8: return launch<T, D, ORD, 8, false>(a, B, st);
    case 16: return launch<T, D, ORD, 16, false>(a, B, st);
    default: return launch<T, D, ORD, 32, false>(a, B, st);
  }
}

template <typename T, int D>
int by_ord(Args<T> a, int ord, long long B, cudaStream_t st) {
  return ord == 2 ? by_k<T, D, 2>(a, B, st) : ord == 1 ? by_k<T, D, 1>(a, B, st) : by_k<T, D, 0>(a, B, st);
}

template <typename T>
int knn_entry(const T* ref, long long ref_bs, const T* nbr, long long nbr_bs, long long B, long long N1, long long N2,
              int D, int k, int ord, int largest, long long S, void* ws, T* vals, long long* inds, void* stream) {
  if (D < 1 || D > 8 || k < 1 || k > 32 || k > N2 || (ord != 0 && ord != 1 && ord != 2) || S < 1 ||
      N2 >= (1LL << 31) || (S > 1 && ws == nullptr))
    return (int)cudaErrorInvalidValue;
  if (B * N1 == 0) return 0;
  Args<T> a{};
  a.ref = ref; a.nbr = nbr; a.ref_bs = ref_bs; a.nbr_bs = nbr_bs; a.N1 = N1; a.N2 = N2; a.S = (int)S; a.k = k;
  a.flip = largest ? Key<T>::MAG : 0;
  a.vals = vals; a.inds = inds;
  a.wkey = reinterpret_cast<typename Key<T>::U*>(ws);
  a.widx = reinterpret_cast<int*>(a.wkey + (S > 1 ? B * N1 * S * round_k(k) : 0));
  cudaStream_t st = (cudaStream_t)stream;
  switch (D) {
    case 1: return by_ord<T, 1>(a, ord, B, st);
    case 2: return by_ord<T, 2>(a, ord, B, st);
    case 3: return by_ord<T, 3>(a, ord, B, st);
    case 4: return by_ord<T, 4>(a, ord, B, st);
    case 5: return by_ord<T, 5>(a, ord, B, st);
    case 6: return by_ord<T, 6>(a, ord, B, st);
    case 7: return by_ord<T, 7>(a, ord, B, st);
    default: return by_ord<T, 8>(a, ord, B, st);
  }
}

template <typename T>
int icp_entry(const T* src, long long src_bs, const T* tgt, long long tgt_bs, const T* pose, long long B, long long N1,
              long long N2, int ord, long long S, void* ws, double* mom, void* stream) {
  if (N2 < 1 || N2 >= (1LL << 31) || (ord != 0 && ord != 1 && ord != 2) || S < 1 || (S > 1 && ws == nullptr))
    return (int)cudaErrorInvalidValue;
  if (B * N1 == 0) return 0;
  Args<T> a{};
  a.ref = src; a.nbr = tgt; a.ref_bs = src_bs; a.nbr_bs = tgt_bs; a.N1 = N1; a.N2 = N2; a.S = (int)S; a.k = 1;
  a.pose = pose; a.mom = mom;
  a.wkey = reinterpret_cast<typename Key<T>::U*>(ws);
  a.widx = reinterpret_cast<int*>(a.wkey + (S > 1 ? B * N1 * S : 0));
  cudaStream_t st = (cudaStream_t)stream;
  return ord == 2 ? launch<T, 3, 2, 1, true>(a, B, st)
       : ord == 1 ? launch<T, 3, 1, 1, true>(a, B, st) : launch<T, 3, 0, 1, true>(a, B, st);
}

}  // namespace knn
}  // namespace b200pose

// the entry points of one dtype (knn.cu: fp32, knn_f64.cu: fp64); B200_EXPORT is defined by the including file
#define KNN_ABI(SFX, CT)                                                                                               \
  B200_EXPORT int b200_knn_##SFX(const CT* ref, long long ref_bstride, const CT* nbr, long long nbr_bstride,          \
                                 long long B, long long N1, long long N2, int D, int k, int ord, int largest,          \
                                 long long splits, void* ws, CT* values, long long* indices, void* stream) {           \
    return knn_entry<CT>(ref, ref_bstride, nbr, nbr_bstride, B, N1, N2, D, k, ord, largest, splits, ws, values,       \
                         indices, stream);                                                                             \
  }                                                                                                                    \
  B200_EXPORT int b200_icp_moments_##SFX(const CT* src, long long src_bstride, const CT* tgt, long long tgt_bstride,  \
                                         const CT* pose, long long B, long long N1, long long N2, int ord,            \
                                         long long splits, void* ws, double* moments, void* stream) {                  \
    return icp_entry<CT>(src, src_bstride, tgt, tgt_bstride, pose, B, N1, N2, ord, splits, ws, moments, stream);      \
  }
