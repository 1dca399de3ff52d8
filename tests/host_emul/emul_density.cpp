// tests/host_emul/emul_density.cpp — CPU build of the density plan (tuna_b200/csrc/density_split.hpp) that tuna_jk_direct and
// tuna_jk_direct_general_dev share: the two maxima of a stack and the run it decides.
#include "../../tuna_b200/csrc/density_split.hpp"

extern "C" void emul_plan_density(const double* P, int nD, int n, double* extrema, int* nDrun, unsigned* anti_mask, double* dens_bound) {
    tuna::density_extrema(P, nD, n, &extrema[0], &extrema[1]);
    const tuna::DensityPlan p = tuna::plan_density(nD, extrema[0], extrema[1]);
    *nDrun = p.nDrun;
    *anti_mask = p.anti_mask;
    *dens_bound = p.dens_bound;
}
