// kmc_metropolis.cuh -- batched independent random-walk Metropolis chains (the reference's `metropolis`,
// src/samplers.jl:9-128) on the device.
//
// One chain is serial; many independent chains are not.  Chain c of a batch is a pure function of (seed, chain id,
// step): its draws are counter-based, so it is the same chain whatever the batch size or launch split.
//
//   metropolis_kernel   fused plugins at their compiled d: one thread per chain, theta / log-density / accept count
//                       in registers for a range of steps [t0, t1) -- proposal, plugin, accept test (:103), update,
//                       thinned store, burn-in counter reset -- and written back once at the end of the launch.
//   mh_propose_kernel   every other plugin, per step: draws + Y = x + sigma .* n ...
//   <density>           ... P1 = plugin(Y) through eval_on_device (FP64, or tcgen05 if the density opted in) ...
//   mh_accept_kernel    ... accept test, update, counters, store.
//   mh_draws_kernel     the normals and uniforms of chains x steps (what a replay of the host loop needs).
//
// Draws of step t (0-based: t = ni + nburnin - 1) of chain id c: Philox4x32-10, key = seed, counter
// (c, t lo, t hi, 0x4D48 << 16 | pair) for pair = 0 .. ceil(d/2)-1; normals 2 pair and 2 pair + 1 are the Box-Muller
// transform of words r0, r1 (philox_normals); the accept uniform is ((r2 & 0xFFFF) << 32 | r3) * 2^-48 of pair 0,
// in [0, 1) like Julia's rand().  The tag keeps these streams apart from emcee's (batch | attempt << 8) and from
// make_theta0s's (0x4D54 << 16).
#pragma once
#include <math_constants.h>

#include "kmc_device.cuh"

namespace kmc {

constexpr unsigned kMhTag = 0x4D480000u;
constexpr int kMhThreads = 256;

struct MhParams {
    double *x;          // [nchains][d] current state (theta0, deep-copied at creation)
    double *lp;         // [nchains] current log-density (p0)
    unsigned *nacc;     // [nchains] accept counters (naccept)
    double *chain_x;    // [ns][nchains][d] sample-major thinned chain (coalesced stores)
    double *chain_lp;   // [ns][nchains]
    const double *rp_n; // replay: normals [steps][nchains][d] from step rp_t0
    const double *rp_u; // replay: accept uniforms [steps][nchains]
    long long rp_t0;
    long long nchains;
    long long t0, t1;   // step range of this launch
    long long nburnin, nthin;
    PhiloxKeys keys;
    unsigned id_base;   // Philox chain id = id_base + local index
};

// Per-component proposal scale, passed by value (constant bank) to the fused kernel.
template <int D>
struct MhSigma {
    double s[D];
};

__device__ __forceinline__ double mh_uniform(const Philox4 &r) {
    return (double)(((unsigned long long)(r.r2 & 0xFFFFu) << 32) | r.r3) * 0x1p-48;  // exact: 48-bit integer * 2^-48
}

// The normals of components [2 pair, 2 pair + 1] of step t of chain id cid (z1 is unused for the last pair of odd d).
__device__ __forceinline__ Philox4 mh_pair(const PhiloxKeys &ks, unsigned cid, unsigned long long t, unsigned pair,
                                           double &z0, double &z1) {
    return philox_normals(ks, cid, (unsigned)t, (unsigned)(t >> 32), kMhTag | pair, z0, z1);
}

// Fused plugins: one thread per chain for steps [t0, t1).
template <template <int> class Dn, int D, bool REPLAY>
static __global__ void __launch_bounds__(kMhThreads) metropolis_kernel(const MhParams p, const Dn<D> dn, const MhSigma<D> sg) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.nchains) return;
    double x[D];
    load_row<D>(p.x + c * D, x);
    double lp = p.lp[c];
    unsigned na = p.nacc[c];
    const unsigned cid = p.id_base + (unsigned)c;
    long long ni = p.t0 + 1 - p.nburnin;  // the reference's loop variable at step t0
    long long ph = ni % p.nthin;
    if (ph < 0) ph += p.nthin;
    long long sidx = ni >= 1 ? (ni - 1) / p.nthin : 0;  // samples stored before ni
    for (long long t = p.t0; t < p.t1; ++t) {
        double y[D], u;
        if constexpr (REPLAY) {
            const size_t slot = (size_t)(t - p.rp_t0) * p.nchains + c;
#pragma unroll
            for (int k = 0; k < D; ++k) y[k] = dadd(x[k], dmul(sg.s[k], __ldcs(p.rp_n + slot * D + k)));
            u = __ldcs(p.rp_u + slot);
        } else {
#pragma unroll
            for (int pr = 0; pr < (D + 1) / 2; ++pr) {
                double z0, z1;
                const Philox4 r = mh_pair(p.keys, cid, (unsigned long long)t, (unsigned)pr, z0, z1);
                if (pr == 0) u = mh_uniform(r);
                y[2 * pr] = dadd(x[2 * pr], dmul(sg.s[2 * pr], z0));  // theta0 .+ sigma .* n: mul, then add
                if (2 * pr + 1 < D) y[2 * pr + 1] = dadd(x[2 * pr + 1], dmul(sg.s[2 * pr + 1], z1));
            }
        }
        const double p1 = dn.logpdf(y);
        if (dsub(p1, lp) > log(u)) {  // :103 strict >, FP64; NaN rejects
#pragma unroll
            for (int k = 0; k < D; ++k) x[k] = y[k];
            lp = p1;
            ++na;
        }
        if (ni > 0 && ph == 0) {
            const size_t o = (size_t)sidx * p.nchains + c;
            store_row_cs<D>(p.chain_x + o * D, x);
            __stcs(p.chain_lp + o, lp);
            ++sidx;
        }
        if (ni == 0) na = 0;  // end of burn-in: only post-burn-in accepts count
        ++ni;
        if (++ph == p.nthin) ph = 0;
    }
    store_row<D>(p.x + c * D, x);
    p.lp[c] = lp;
    p.nacc[c] = na;
}

// Batched plugins, stage 1 of a step: Y = x + sigma .* n and the accept uniform.  One thread per (chain, pair).
template <bool REPLAY>
static __global__ void __launch_bounds__(256) mh_propose_kernel(const MhParams p, const double *__restrict__ sigma, long long t,
                                                                int d, double *__restrict__ Y, double *__restrict__ U) {
    const int npair = (d + 1) / 2;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.nchains * npair) return;
    const long long c = e / npair;
    const int pr = (int)(e - c * npair), k = 2 * pr;
    const double *xc = p.x + c * d;
    double *yc = Y + c * d;
    double z0, z1, u = 0.0;
    if constexpr (REPLAY) {
        const size_t slot = (size_t)(t - p.rp_t0) * p.nchains + c;
        z0 = __ldcs(p.rp_n + slot * d + k);
        z1 = k + 1 < d ? __ldcs(p.rp_n + slot * d + k + 1) : 0.0;
        if (pr == 0) u = __ldcs(p.rp_u + slot);
    } else {
        const Philox4 r = mh_pair(p.keys, p.id_base + (unsigned)c, (unsigned long long)t, (unsigned)pr, z0, z1);
        if (pr == 0) u = mh_uniform(r);
    }
    yc[k] = dadd(xc[k], dmul(sigma[k], z0));
    if (k + 1 < d) yc[k + 1] = dadd(xc[k + 1], dmul(sigma[k + 1], z1));
    if (pr == 0) U[c] = u;
}

// Batched plugins, stage 3 of a step: one warp per chain, lanes stride over the components.
static __global__ void __launch_bounds__(256) mh_accept_kernel(const MhParams p, const double *__restrict__ Y,
                                                               const double *__restrict__ P1, const double *__restrict__ U,
                                                               int d, long long ni, int store, long long sidx) {
    const long long c = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned lane = threadIdx.x & 31;
    if (c >= p.nchains) return;
    const double p1 = P1[c], p0 = p.lp[c];
    const bool acc = dsub(p1, p0) > log(U[c]);  // :103
    double *xc = p.x + c * d;
    const double *yc = Y + c * d;
    if (acc)
        for (int k = lane; k < d; k += 32) xc[k] = yc[k];
    if (store) {
        const size_t o = (size_t)sidx * p.nchains + c;
        for (int k = lane; k < d; k += 32) __stcs(p.chain_x + o * d + k, acc ? yc[k] : xc[k]);
        if (lane == 0) __stcs(p.chain_lp + o, acc ? p1 : p0);
    }
    if (lane == 0) {
        if (acc) {
            p.lp[c] = p1;
            p.nacc[c] += 1u;
        }
        if (ni == 0) p.nacc[c] = 0u;
    }
}

// normals [t][c][d] and uniforms [t][c] of chains [chain0, chain0 + nchains), steps [t0, t0 + nsteps).
static __global__ void mh_draws_kernel(PhiloxKeys ks, unsigned chain0, long long nchains, long long t0, long long nsteps, int d,
                                       double *__restrict__ normals, double *__restrict__ u) {
    const int npair = (d + 1) / 2;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nsteps * nchains * npair) return;
    const long long row = e / npair;  // = ts * nchains + c
    const int pr = (int)(e - row * npair);
    const long long ts = row / nchains, c = row - ts * nchains;
    double z0, z1;
    const Philox4 r = mh_pair(ks, chain0 + (unsigned)c, (unsigned long long)(t0 + ts), (unsigned)pr, z0, z1);
    normals[row * d + 2 * pr] = z0;
    if (2 * pr + 1 < d) normals[row * d + 2 * pr + 1] = z1;
    if (pr == 0) u[row] = mh_uniform(r);
}

}  // namespace kmc
