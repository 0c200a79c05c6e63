// knn.cu — C-ABI of the k-nearest-neighbour search and the ICP step for fp32, and the split planner (kernels: knn.cuh).
// The fp64 entry points are compiled in knn_f64.cu so that the two instantiation sets build in parallel.
#include "knn.cuh"
#include "b200pose.h"   // every definition is checked against the generated declaration

#define B200_EXPORT extern "C" __attribute__((visibility("default")))

using namespace b200pose::knn;

B200_EXPORT long long b200_knn_plan(long long B, long long N1, long long N2, int k, int elem_size, int sms,
                                    long long* splits) {
  return plan(B, N1, N2, k, elem_size, sms, splits);
}

KNN_ABI(f32, float)
