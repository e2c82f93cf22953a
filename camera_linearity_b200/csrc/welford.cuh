// K3 helpers shared by the 8-bit (welford.cu) and 16-bit (welford_u16.cu) Welford kernels.
#pragma once

#include "common.cuh"

namespace cl {
namespace {

// ---- exact sequential recurrence ------------------------------------------------------------------
struct WelfordState {
    double mean, m2;
};

// video_processing.py:205-208 with n as a double and rn = RN(1/n)
__device__ __forceinline__ void welford_step(WelfordState& s, double x, double n, double rn) {
    const double delta = __dsub_rn(x, s.mean);
    const double q0 = __dmul_rn(delta, rn);
    const double rem = __fma_rn(-q0, n, delta);
    const double q = __fma_rn(rem, rn, q0);          // == RN(delta / n)
    s.mean = __dadd_rn(s.mean, q);
    s.m2 = __dadd_rn(s.m2, __dmul_rn(delta, __dsub_rn(x, s.mean)));
}

__device__ __forceinline__ void welford_mean_step(double& mean, double x, double n, double rn) {
    const double delta = __dsub_rn(x, mean);          // welford_step without M2 (the replay only decides the mean)
    const double q0 = __dmul_rn(delta, rn);
    const double rem = __fma_rn(-q0, n, delta);
    mean = __dadd_rn(mean, __fma_rn(rem, rn, q0));
}

// Head of the stack form's workspace, followed by the tie list (one uint32 sample index per sample).
// dn_out_of_range: set by the 16-bit ICRF kernels when a DN has no row in a table shorter than 65536 rows.
struct StackHeader {
    unsigned int tie_count;
    unsigned int dn_out_of_range;
    unsigned int pad[2];
};

inline unsigned grid_for(int64_t items, int threads, int per_sm) {
    int64_t b = (items + threads - 1) / threads;
    const int64_t cap = (int64_t)sm_count() * per_sm;
    if (b > cap) b = cap;
    return (unsigned)(b < 1 ? 1 : b);
}

}  // namespace
}  // namespace cl
