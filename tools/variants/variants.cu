// DEV ONLY (not part of the package): candidate configurations of the v2 shell for the headline kernels, built into
// tools/variants/libvariants.so by tools/variants/build.sh and timed by tools/variants/ab.py.
// NAME = <op>_<dtype>_s<S>o<OS>_pf<PF>: S input / OS output stages, PF tiles hinted into L2 before the dependency
// wait.  The grid policy is the shipped launcher's (B200POSE_PDL / B200POSE_CTAS_PER_SM apply).
#include "lie_kernels.cuh"
using namespace b200pose;
#define VAR(OPN, OPT, CT, SFX, S, OS, PF)                                                                          \
  extern "C" __attribute__((visibility("default"))) int OPN##_##SFX##_s##S##o##OS##_pf##PF(                        \
      const CT* i0, CT* o0, long long n, void* st) {                                                               \
    const CT* in[1] = {i0}; CT* out[1] = {o0};                                                                     \
    return launch_stream_tma<OPT<SE3g, CT>, S, OS, kThreads, 1, PF>(in, out, n, (cudaStream_t)st);                \
  }
#define PAIR(CT, SFX, S, OS, PF) VAR(exp, OpExpFwd, CT, SFX, S, OS, PF) VAR(log, OpLogFwd, CT, SFX, S, OS, PF)
PAIR(float, f32, 3, 2, 0)    // no hint
PAIR(float, f32, 3, 2, 3)    // the shipped fp32 configuration
PAIR(float, f32, 3, 2, 6)
PAIR(float, f32, 3, 1, 3)
PAIR(float, f32, 3, 1, 6)
PAIR(float, f32, 2, 1, 2)
PAIR(float, f32, 4, 1, 4)
PAIR(double, f64, 2, 2, 0)
PAIR(double, f64, 2, 2, 2)   // the shipped fp64 configuration
PAIR(double, f64, 2, 1, 2)
