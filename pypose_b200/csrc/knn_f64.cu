// knn_f64.cu — fp64 C-ABI of the k-nearest-neighbour search and the ICP step (kernels: knn.cuh).
#include "knn.cuh"
#include "b200pose.h"   // every definition is checked against the generated declaration

#define B200_EXPORT extern "C" __attribute__((visibility("default")))

using namespace b200pose::knn;

KNN_ABI(f64, double)
