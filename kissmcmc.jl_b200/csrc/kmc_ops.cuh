// kmc_ops.cuh -- the kernel registry of the fused thread-per-walker plugins: one Ops record per (plugin, d) with the
// entry points of every kernel family compiled for it.  The instantiations live in their own translation units
// (kmc_ops_*.cu) so that the library builds in parallel; kmc_api.cu only looks records up.
#pragma once
#include <cstddef>

namespace kmc_host {

// How a plugin evaluates its log-density; the values are what kmc_density_get_info("batched") reports.  BATCH_FUSED is 0,
// so `if (ops.batch)` reads "a batched plugin".
enum Batch : int {
    BATCH_FUSED = 0,     // fused thread-per-walker kernels
    BATCH_GAUSSIAN = 1,  // dense Gaussian contraction (kmc_batched.cuh; tcgen05 in kmc_tc.cuh)
    BATCH_LOGISTIC = 2,  // logistic regression over a data set
    BATCH_EXP = 3,       // exponential at a d with no fused kernel: thread-per-point sum
};

struct Ops {
    const void *run[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [replay][smem-resident state]
    const void *run_peer = nullptr;  // general kernel with cross-GPU partner gathers (Philox mode)
    const void *run_bulk[2] = {nullptr, nullptr};  // [peer] bulk (TMA) general kernel, Philox mode, even D >= 6
    size_t bulk_smem = 0;
    const void *run_push = nullptr;  // sharded ensemble with owner-computes pushes (kmc_push.cuh), Philox mode, even D
    size_t smem_per_walker = 0;  // bytes of shared memory per owned walker (SMEM mode)
    int block = 0;               // max threads per CTA of the run kernels
    int min_blocks = 1;          // CTAs per SM the kernels are compiled for
    Batch batch = BATCH_FUSED;
    const void *eval = nullptr;
    const void *mh[2] = {nullptr, nullptr};  // [replay] metropolis_kernel (kmc_metropolis.cuh)
    const void *mh_chol[2] = {nullptr, nullptr};  // [replay] metropolis_chol_kernel: correlated proposal
    size_t dn_bytes = 0;
    int nparams = 0;
};


// (plugin, d) -> Ops; false if no kernel is compiled for that dimension.
bool ops_exponential(int d, Ops &o);
bool ops_gaussian(int d, Ops &o);     // the fused FP64 Gaussian, d <= 16
bool ops_rosenbrock(int d, Ops &o);
bool ops_lognormal(int d, Ops &o);

}  // namespace kmc_host

#ifdef KMC_OPS_IMPL  // only the kmc_ops_*.cu translation units instantiate kernels
#include "kmc_kernels.cuh"
#include "kmc_push.cuh"
#include "kmc_metropolis.cuh"

namespace kmc_host {

template <template <int> class Dn, int D>
Ops make_ops() {
    Ops o;
    o.run[0][0] = (const void *)kmc::emcee_run_kernel<Dn, D, false>;
    o.run[1][0] = (const void *)kmc::emcee_run_kernel<Dn, D, true>;
    o.run_peer = (const void *)kmc::emcee_run_kernel<Dn, D, false, true>;
    if constexpr (D % 2 == 0 && D >= 6) {
        o.run_bulk[0] = (const void *)kmc::emcee_bulk_kernel<Dn, D, false>;
        o.run_bulk[1] = (const void *)kmc::emcee_bulk_kernel<Dn, D, true>;
        o.bulk_smem = (size_t)3 * kmc::kBulkThreads * D * 8 + 16;
    }
    if constexpr (D % 2 == 0) {
        o.run_push = (const void *)kmc::emcee_push_kernel<Dn, D>;
    }
    if (D <= 4) {  // shared-memory-resident variant for small rows
        o.run[0][1] = (const void *)kmc::emcee_smem_kernel<Dn, (D <= 4 ? D : 1), false>;
        o.run[1][1] = (const void *)kmc::emcee_smem_kernel<Dn, (D <= 4 ? D : 1), true>;
    }
    o.smem_per_walker = 8 * D + 8 + 4;
    o.block = kmc::max_threads<D>();
    o.min_blocks = kmc::min_blocks<D>();
    o.eval = (const void *)kmc::density_eval_kernel<Dn, D>;
    o.mh[0] = (const void *)kmc::metropolis_kernel<Dn, D, false>;
    o.mh[1] = (const void *)kmc::metropolis_kernel<Dn, D, true>;
    o.mh_chol[0] = (const void *)kmc::metropolis_chol_kernel<Dn, D, false>;
    o.mh_chol[1] = (const void *)kmc::metropolis_chol_kernel<Dn, D, true>;
    o.dn_bytes = sizeof(Dn<D>);
    o.nparams = Dn<D>::nparams;
    return o;
}

template <template <int> class Dn>
bool ops_for_dim(int d, Ops &o) {
    switch (d) {
        case 2: o = make_ops<Dn, 2>(); return true;
        case 10: o = make_ops<Dn, 10>(); return true;
#ifndef KMC_FAST_BUILD  // experiment builds (build/variants/) compile d = 2 and d = 10 only
        case 1: o = make_ops<Dn, 1>(); return true;
        case 3: o = make_ops<Dn, 3>(); return true;
        case 4: o = make_ops<Dn, 4>(); return true;
        case 5: o = make_ops<Dn, 5>(); return true;
        case 6: o = make_ops<Dn, 6>(); return true;
        case 8: o = make_ops<Dn, 8>(); return true;
        case 12: o = make_ops<Dn, 12>(); return true;
        case 16: o = make_ops<Dn, 16>(); return true;
#endif
        default: return false;
    }
}

}  // namespace kmc_host
#endif
