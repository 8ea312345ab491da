// Kernel instantiations of the fused "gaussian_mixture" plugin, d in {1..6, 8, 10, 12, 16}.
#define KMC_OPS_IMPL
#include "kmc_ops.cuh"

namespace kmc_host {
bool ops_gaussian_mixture(int d, Ops &o) { return ops_for_dim<kmc::GaussianMixture>(d, o); }
}  // namespace kmc_host
