// sim_terms.cuh — the per-pair update and the final formula of the exact similarities (core/sim.go), shared by the
// sparse Fit (sim_stream.cu) and the similarity row of a query given as a rating list (given.cu), so that both
// apply the reference's IEEE operations in the same way.  The library is built with --fmad=false.
//
// Accumulators of a pair live at acc[j], acc[JC + j], acc[2 * JC + j] (and acc[3 * JC + j] with SHRINK):
//   MSD      sum of (ra - rb)^2, count
//   others   sum of ra^2, sum of rb^2, sum of ra * rb (and the co-rating count for the shrinkage)
// ra is the a-side term (the rating, or the rating minus the row's Pearson mean / baseline), rb the b-side term.
#pragma once

#include "common.cuh"

template <int SIM, bool SHRINK, int JC>
__device__ __forceinline__ void stream_update(double *acc, int j, double ra, double raa, double rb) {
    if (SIM == RS_SIM_MSD) {
        const double d = ra - rb;
        acc[j] += d * d;                 // sum += (ir-jr)^2   core/sim.go:37
        acc[JC + j] += 1.0;              // count++            core/sim.go:38
    } else {
        acc[j] += raa;                   // m += ..            core/sim.go:19 / :75
        acc[JC + j] += rb * rb;          // n += rb*rb         core/sim.go:20 / :76
        acc[2 * JC + j] += ra * rb;      // l += ra*rb         core/sim.go:21 / :77
        if (SHRINK) acc[3 * JC + j] += 1.0;
    }
}

// The similarity of one pair from its accumulators acc[0], acc[stride], acc[2 * stride] (and acc[3 * stride] with
// SHRINK), as above; acc[2 * stride] is not read by MSD.  No term at all gives 0 / 0 = NaN, the reference's value for
// a pair without a co-rating.
template <int SIM, bool SHRINK>
__device__ __forceinline__ double sim_value(const double *acc, int stride, double shrinkage) {
    double s;
    if (SIM == RS_SIM_MSD) s = 1.0 / (acc[0] / acc[stride] + 1.0);                      // core/sim.go:43
    else s = acc[2 * stride] / (sqrt(acc[0]) * sqrt(acc[stride]));                      // core/sim.go:24 / :80
    if (SHRINK) {
        const double cn = acc[3 * stride];
        s = (cn - 1.0) / (cn - 1.0 + shrinkage) * s;
    }
    return s;
}
