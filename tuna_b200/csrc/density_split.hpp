// density_split.hpp — which densities a direct build runs for a density stack of any real P (host densities: stage_host_density,
// device densities: tuna_jk_direct_general_dev / tuna_jk_direct_group_general_dev, both in tuna_b200.cu).
//
// J[P] = J[S] and K[P] = K[S] + K[A] for S = (P + P^T) / 2 and A = (P - P^T) / 2, K[A] antisymmetric.  SCF densities are symmetric to
// round-off (reference guess densities are not always: asymmetry ~1e-8 was observed); a stack with max|P - P^T| > 1e-15 max|P| runs as
// 2 nD densities, S first, the A parts marked in anti_mask.  Plain C++: the tests compile it for the host.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstddef>

namespace tuna {

struct DensityPlan {
    int nDrun;              // densities the build runs: nD, or 2 nD for a split stack
    unsigned anti_mask;     // bit d: density d of the run is antisymmetric
    double dens_bound;      // the bound the cached job lists are pre-screened with (tuna_ctx::dens_bound)
};

// pmax = max|P|, amax = max|P - P^T| over the whole stack.  Both are maxima, hence exact: a device scan of the same stack gives the same
// two numbers, and the same plan.
inline DensityPlan plan_density(int nD, double pmax, double amax) {
    const bool general = amax > 1e-15 * pmax;
    DensityPlan p;
    p.nDrun = general ? 2 * nD : nD;
    p.anti_mask = general ? ((1u << nD) - 1u) << nD : 0u;
    p.dens_bound = std::max(1e3, 1e3 * pmax);       // static pre-screening stays below the device's exact density-weighted test
    return p;
}

// The two maxima of a host stack of nD n x n densities.
inline void density_extrema(const double* P, int nD, int n, double* pmax, double* amax) {
    const size_t nn = (size_t)n * n;
    double pm = 0.0, am = 0.0;
    for (int d = 0; d < nD; ++d)
        for (int i = 0; i < n; ++i)
            for (int j = 0; j <= i; ++j) {
                const double x = P[d * nn + (size_t)i * n + j], y = P[d * nn + (size_t)j * n + i];
                pm = std::max(pm, std::max(std::fabs(x), std::fabs(y)));
                am = std::max(am, std::fabs(x - y));
            }
    *pmax = pm;
    *amax = am;
}

}  // namespace tuna
