// kmc_metropolis.cuh -- batched independent random-walk Metropolis chains (the reference's `metropolis`,
// src/samplers.jl:9-128) on the device.
//
// One chain is serial; many independent chains are not.  Chain c of a batch is a pure function of (seed, chain id,
// step): its draws are counter-based, so it is the same chain whatever the batch size or launch split.
//
//   metropolis_kernel   fused plugins at their compiled d: one thread per chain, theta / log-density / accept count
//                       in registers for a range of steps [t0, t1) -- proposal, plugin, accept test (:103), update,
//                       thinned store, burn-in counter reset -- and written back once at the end of the launch.
//   metropolis_chol_kernel  the same loop with the correlated proposal Y = x + L z (L lower-triangular, by value).
//   mh_propose_kernel   every other plugin, per step: draws + Y = x + sigma .* n ...
//     (correlated:      mh_normals_kernel draws Z and U, then mh_chol_kernel forms Y = X + L Z)
//   <density>           ... P1 = plugin(Y) through eval_on_device (FP64, or tcgen05 if the density opted in) ...
//   mh_accept_kernel    ... accept test, update, counters, store.
//   mh_draws_kernel     the normals and uniforms of chains x steps (what a replay of the host loop needs).
//
// The correlated proposal's arithmetic, which the CPU oracle restates bit for bit: for i = 0 .. d-1,
// s = 0.0; s = s + L[i][j] * z[j] for j = 0 .. i ascending (mul, then add; never an FMA); y[i] = x[i] + s.
// With L = diag(sigma) this is bit-identical to x + sigma .* z: the added products are signed zeros.
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

// Lower-triangular Cholesky factor, packed by rows: L[i][j] (j <= i) at i (i + 1) / 2 + j.  By value, like MhSigma.
template <int D>
struct MhChol {
    double l[D * (D + 1) / 2];
};

// The fused kernels' arguments (MhParams, the plugin, the proposal) share the 4 KB kernel-parameter space.
template <class Dn, class Prop>
struct MhParamsFit {
    static constexpr bool value = sizeof(MhParams) + sizeof(Dn) + sizeof(Prop) <= 4096;
};

__device__ __forceinline__ double mh_uniform(const Philox4 &r) {
    return (double)(((unsigned long long)(r.r2 & 0xFFFFu) << 32) | r.r3) * 0x1p-48;  // exact: 48-bit integer * 2^-48
}

// The normals of components [2 pair, 2 pair + 1] of step t of chain id cid (z1 is unused for the last pair of odd d).
__device__ __forceinline__ Philox4 mh_pair(const PhiloxKeys &ks, unsigned cid, unsigned long long t, unsigned pair,
                                           double &z0, double &z1) {
    return philox_normals(ks, cid, (unsigned)t, (unsigned)(t >> 32), kMhTag | pair, z0, z1);
}

// Components k, k + 1 (k even; k + 1 skipped at D) of the proposal from the normals z0, z1 of pair k / 2.
template <int D>
__device__ __forceinline__ void mh_propose_pair(const MhSigma<D> &sg, const double *x, double *y, int k, double z0,
                                                double z1) {
    y[k] = dadd(x[k], dmul(sg.s[k], z0));  // theta0 .+ sigma .* n: mul, then add
    if (k + 1 < D) y[k + 1] = dadd(x[k + 1], dmul(sg.s[k + 1], z1));
}

// Correlated: y[i] (i > k + 1) holds the partial sum over j < k of row i until its own pair comes.  Pairs arrive in
// ascending order, z0 before z1, so every row adds its products in ascending j.
template <int D>
__device__ __forceinline__ void mh_propose_pair(const MhChol<D> &ch, const double *x, double *y, int k, double z0,
                                                double z1) {
    if (k == 0) {
#pragma unroll
        for (int i = 0; i < D; ++i) y[i] = 0.0;
    }
#pragma unroll
    for (int i = k; i < D; ++i) y[i] = dadd(y[i], dmul(ch.l[i * (i + 1) / 2 + k], z0));
#pragma unroll
    for (int i = k + 1; i < D; ++i) y[i] = dadd(y[i], dmul(ch.l[i * (i + 1) / 2 + k + 1], z1));
    y[k] = dadd(x[k], y[k]);
    if (k + 1 < D) y[k + 1] = dadd(x[k + 1], y[k + 1]);
}

template <class Prop>
struct MhIsChol {
    static constexpr bool value = false;
};
template <int D>
struct MhIsChol<MhChol<D>> {
    static constexpr bool value = true;
};

// Fused plugins: one thread per chain for steps [t0, t1).  Prop is MhSigma<D> (y = x + sigma .* z) or MhChol<D>
// (y = x + L z, formed pair by pair as the Philox pairs arrive: y[i] needs only z[0 .. i]).
template <template <int> class Dn, int D, bool REPLAY, class Prop>
__device__ __forceinline__ void metropolis_chain(const MhParams &p, const Dn<D> &dn, const Prop &sg) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.nchains) return;
    double x[D];
    load_row<D>(p.x + c * D, x);
    double lp = p.lp[c];
    unsigned na = p.nacc[c];
    const unsigned cid = p.id_base + (unsigned)c;
    // the reference's loop variable at step t0, its phase and the samples stored before it; the loop below advances its
    // own copy (ThinClock::advance here does not compile to the same code)
    const ThinClock<> clk0 = ThinClock<>::at(p.t0, p.nburnin, p.nthin);
    long long ni = clk0.n, ph = clk0.phase, sidx = clk0.sidx;
    for (long long t = p.t0; t < p.t1; ++t) {
        double y[D], u;
        if constexpr (REPLAY) {
            const size_t slot = (size_t)(t - p.rp_t0) * p.nchains + c;
            if constexpr (MhIsChol<Prop>::value) {
#pragma unroll
                for (int k = 0; k < D; k += 2)
                    mh_propose_pair<D>(sg, x, y, k, __ldcs(p.rp_n + slot * D + k),
                                       k + 1 < D ? __ldcs(p.rp_n + slot * D + k + 1) : 0.0);
            } else {
#pragma unroll
                for (int k = 0; k < D; ++k) y[k] = dadd(x[k], dmul(sg.s[k], __ldcs(p.rp_n + slot * D + k)));
            }
            u = __ldcs(p.rp_u + slot);
        } else {
#pragma unroll
            for (int pr = 0; pr < (D + 1) / 2; ++pr) {
                double z0, z1;
                const Philox4 r = mh_pair(p.keys, cid, (unsigned long long)t, (unsigned)pr, z0, z1);
                if (pr == 0) u = mh_uniform(r);
                mh_propose_pair<D>(sg, x, y, 2 * pr, z0, z1);
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

template <template <int> class Dn, int D, bool REPLAY>
static __global__ void __launch_bounds__(kMhThreads) metropolis_kernel(const MhParams p, const Dn<D> dn, const MhSigma<D> sg) {
    static_assert(MhParamsFit<Dn<D>, MhSigma<D>>::value, "kernel parameters of metropolis_kernel exceed 4 KB");
    metropolis_chain<Dn, D, REPLAY>(p, dn, sg);
}

template <template <int> class Dn, int D, bool REPLAY>
static __global__ void __launch_bounds__(kMhThreads) metropolis_chol_kernel(const MhParams p, const Dn<D> dn,
                                                                            const MhChol<D> ch) {
    static_assert(MhParamsFit<Dn<D>, MhChol<D>>::value, "kernel parameters of metropolis_chol_kernel exceed 4 KB");
    metropolis_chain<Dn, D, REPLAY>(p, dn, ch);
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

// Batched plugins with a correlated proposal, stage 1a: the normals Z [nchains][d] and the accept uniform of step t.
template <bool REPLAY>
static __global__ void __launch_bounds__(256) mh_normals_kernel(const MhParams p, long long t, int d,
                                                                double *__restrict__ Z, double *__restrict__ U) {
    const int npair = (d + 1) / 2;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.nchains * npair) return;
    const long long c = e / npair;
    const int pr = (int)(e - c * npair), k = 2 * pr;
    double *zc = Z + c * d;
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
    zc[k] = z0;
    if (k + 1 < d) zc[k + 1] = z1;
    if (pr == 0) U[c] = u;
}

// Stage 1b: Y = X + L Z, L [d][d] row-major lower-triangular.  A CTA owns kMhTri rows i x kMhTri chains; thread
// (tx, ty) owns row i0 + tx of chains c0 + ty + 8 r.  It walks the k-tiles up to its diagonal in ascending order with
// no split-K, so every output adds its products in the order of the proposal contract (s = 0; s += L[i][j] z[j] for
// j = 0 .. i; y = x + s), and skips the tiles above the diagonal.
constexpr int kMhTri = 32;
static __global__ void __launch_bounds__(256) mh_chol_kernel(const double *__restrict__ X, const double *__restrict__ L,
                                                             const double *__restrict__ Z, long long nchains, int d,
                                                             double *__restrict__ Y) {
    constexpr int R = kMhTri / 8;
    __shared__ double Ls[kMhTri][kMhTri + 1], Zs[kMhTri][kMhTri + 1];
    const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * kMhTri + tx;
    const int i0 = blockIdx.y * kMhTri, i = i0 + tx;  // chain tiles on x: grid.y (<= 65535) only counts row tiles
    const long long c0 = (long long)blockIdx.x * kMhTri;
    double s[R];
#pragma unroll
    for (int r = 0; r < R; ++r) s[r] = 0.0;
    for (int j0 = 0; j0 <= i0; j0 += kMhTri) {
        for (int e = tid; e < kMhTri * kMhTri; e += 256) {  // coalesced along j
            const int a = e / kMhTri, b = e % kMhTri;
            Ls[a][b] = (i0 + a < d && j0 + b < d) ? L[(size_t)(i0 + a) * d + j0 + b] : 0.0;
            Zs[a][b] = (c0 + a < nchains && j0 + b < d) ? Z[(c0 + a) * d + j0 + b] : 0.0;
        }
        __syncthreads();
        const int jn = min(kMhTri, i - j0 + 1);  // j <= i: the diagonal tile stops at the thread's own row
        for (int jj = 0; jj < jn; ++jj) {
            const double l = Ls[tx][jj];
#pragma unroll
            for (int r = 0; r < R; ++r) s[r] = dadd(s[r], dmul(l, Zs[ty + 8 * r][jj]));
        }
        __syncthreads();
    }
    if (i >= d) return;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const long long c = c0 + ty + 8 * r;
        if (c < nchains) Y[c * d + i] = dadd(X[c * d + i], s[r]);
    }
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

// Covariance of the stored chain (kmc_emcee_chain_covariance): the nrows rows of chain [nrows][d], shifted by row 0
// like chain_moments_kernel, with a constant column v[d] = 1 appended so that one upper triangle over d + 1 columns
// holds both sum(v_a v_b) and sum(v_a).  A fixed grid of kCovGrid CTAs each reduces a fixed contiguous row range into
// its own partials, and mh_cov_final_kernel adds the partials of the CTAs in ascending order: no atomics, so the
// result's bits depend only on the stored chain.
constexpr int kCovMaxD = 128, kCovGrid = 256, kCovThreads = 256, kCovRows = 16;
constexpr int kCovPerThread = ((kCovMaxD + 1) * (kCovMaxD + 2) / 2 + kCovThreads - 1) / kCovThreads;

static __global__ void __launch_bounds__(kCovThreads) mh_cov_partial_kernel(const double *__restrict__ chain,
                                                                            long long nrows, int d,
                                                                            double *__restrict__ part /* [grid][P] */) {
    __shared__ double V[kCovRows][kCovMaxD + 1];
    const int dc = d + 1, P = dc * (dc + 1) / 2;
    short ia[kCovPerThread], ib[kCovPerThread];
    double acc[kCovPerThread];
#pragma unroll
    for (int k = 0; k < kCovPerThread; ++k) {  // entry e -> (a, b), a <= b, row-major upper triangle
        int e = threadIdx.x + k * kCovThreads, a = 0;
        if (e >= P) e = 0;
        while (e >= dc - a) e -= dc - a++;
        ia[k] = (short)a;
        ib[k] = (short)(a + e);
        acc[k] = 0.0;
    }
    const long long r0 = nrows * blockIdx.x / gridDim.x, r1 = nrows * (blockIdx.x + 1) / gridDim.x;
    for (long long rb = r0; rb < r1; rb += kCovRows) {
        const int nr = (int)min((long long)kCovRows, r1 - rb);
        for (int e = threadIdx.x; e < nr * dc; e += kCovThreads) {
            const int r = e / dc, a = e - r * dc;
            V[r][a] = a < d ? chain[(rb + r) * d + a] - chain[a] : 1.0;
        }
        __syncthreads();
        for (int r = 0; r < nr; ++r) {
#pragma unroll
            for (int k = 0; k < kCovPerThread; ++k)  // the guard is uniform: small d skips the unused slots
                if (k * kCovThreads < P) acc[k] = fma(V[r][ia[k]], V[r][ib[k]], acc[k]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int k = 0; k < kCovPerThread; ++k) {
        const int e = threadIdx.x + k * kCovThreads;
        if (e < P) part[(size_t)blockIdx.x * P + e] = acc[k];
    }
}

static __global__ void mh_cov_final_kernel(const double *__restrict__ part, int P, int ngrid, double *__restrict__ out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= P) return;
    double s = 0.0;
    for (int g = 0; g < ngrid; ++g) s += part[(size_t)g * P + e];
    out[e] = s;
}

}  // namespace kmc
