// kmc_batched.cuh -- the half-step as a three-kernel pipeline for log-densities that are
// dense contractions over the whole active half (d up to 128 Gaussian: [W x d]·[d x d];
// logistic regression: [W x d]·[d x N] + row reduction):
//
//   propose_kernel   draws (src/samplers.jl:250,:252,:260) + proposal y = xj + z(xk - xj) (:255)
//                    for every active walker of this shard -> Y [W][d], z, u
//   <density>        logp1[W] = plugin(Y)  (:257)   FP64 CUDA-core kernels here; the tcgen05
//                    kernels (kmc_tc.cuh) replace exactly this stage
//   accept_kernel    accept test (:260), state update (:261-265), thinned chain store (:268-272),
//                    burn-in counter reset (:285-288)
//
// The same density kernels serve kmc_density_eval (initial p0s :209, make_theta0s :334-338).
#pragma once
#include <cuda_bf16.h>

#include "kmc_kernels.cuh"

namespace kmc {

struct BatchBuf {
    double *Y;    // [W][d] proposals of the active walkers of this shard
    double *z;    // [W]
    double *u;    // [W]
    double *p1;   // [W] log-density of the proposals
    unsigned *j;  // [W] partner index (global), kept for the recomputing accept stage
};

// One warp per active walker; lanes stride over the components (coalesced row access).
template <bool REPLAY>
static __global__ void __launch_bounds__(256) propose_kernel(const RunParams p, const BatchBuf b, long long h, int d) {
    const unsigned w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const unsigned W = p.shard_end - p.shard_begin;
    if (w >= W) return;
    const unsigned i = p.shard_begin + w;
    const unsigned batch = (unsigned)(h & 1);
    unsigned j;
    double z, u;
    step_draws<REPLAY>(p, h, i, j, z, u);
    const double *xk = p.x + ((size_t)(batch ? p.nhalf : 0u) + i) * d;
    const double *xj = p.x + (size_t)j * d;
    double *y = b.Y + (size_t)w * d;
    for (int c = lane; c < d; c += 32) y[c] = stretch_coord(xj[c], xk[c], z);  // :255
    if (lane == 0) {
        b.z[w] = z;
        b.u[w] = u;
    }
}

template <bool REPLAY>
static __global__ void __launch_bounds__(256) accept_kernel(const RunParams p, const BatchBuf b, long long h, int d,
                                                     long long n, int store, long long sidx) {
    const unsigned w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const unsigned W = p.shard_end - p.shard_begin;
    if (w >= W) return;
    const unsigned i = p.shard_begin + w;
    const unsigned batch = (unsigned)(h & 1);
    const size_t k = (size_t)(batch ? p.nhalf : 0u) + i;
    const double p1 = b.p1[w], p0 = p.lp[k];
    const bool acc = accept_exact<false>(p.nm1, b.z[w], p1, p0, b.u[w]);  // :260 (exact FP64; once per walker)
    double *xk = p.x + k * d;
    const double *y = b.Y + (size_t)w * d;
    if (acc)  // :261-265
        for (int c = lane; c < d; c += 32) xk[c] = y[c];
    __syncwarp();
    if (lane == 0) {
        if (acc) {
            p.lp[k] = p1;
            p.nacc[k] += 1u;
        }
        if (batch == 1 && n == 0) {  // :285-288 (both halves of this walker position)
            p.nacc[i] = 0u;
            p.nacc[(size_t)p.nhalf + i] = 0u;
        }
    }
    if (store) {  // :268-272
        const size_t o = chain_row(p, sidx, batch, i);
        for (int c = lane; c < d; c += 32) __stcs(p.chain_x + o * d + c, acc ? y[c] : xk[c]);
        if (lane == 0) __stcs(p.chain_lp + o, acc ? p1 : p0);
    }
}

// Variants for the tcgen05 Gaussian path: the proposal is never written in FP64.  propose emits the
// centred proposal (y - mu) already split into three bf16 pieces [3][wpad][128] (what the GEMM's
// TMA loads); accept recomputes y = xj + z(xk - xj) -- the same three IEEE operations, so the same
// bits -- only for accepted walkers (and for the chain store).  Saves the Y write, the Y read of a
// separate split kernel and the Y read of accept: ~230 MB -> ~120 MB per half-step at d = 100.
template <bool REPLAY>
static __global__ void __launch_bounds__(256) propose_pieces_kernel(const RunParams p, const BatchBuf b, long long h, int d,
                                                             const double *__restrict__ mu,
                                                             __nv_bfloat16 *__restrict__ pieces, long long wpad) {
    const unsigned w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= wpad) return;
    const unsigned W = p.shard_end - p.shard_begin;
    const size_t plane = (size_t)wpad * 128;
    __nv_bfloat16 *row = pieces + (size_t)w * 128;
    if (w >= W) {  // padding rows of the last tile
        for (int c = lane; c < 128; c += 32)
            for (int pc = 0; pc < 3; ++pc) row[pc * plane + c] = __float2bfloat16(0.0f);
        return;
    }
    const unsigned i = p.shard_begin + w;
    const unsigned batch = (unsigned)(h & 1);
    unsigned j;
    double z, u;
    step_draws<REPLAY>(p, h, i, j, z, u);
    const double *xk = p.x + ((size_t)(batch ? p.nhalf : 0u) + i) * d;
    const double *xj = p.x + (size_t)j * d;
    for (int c = 2 * lane; c < 128; c += 64) {  // column pairs: one 4-byte store per piece
        double v0 = 0.0, v1 = 0.0;
        if (c < d) v0 = stretch_coord(xj[c], xk[c], z) - mu[c];  // :255, centred
        if (c + 1 < d) v1 = stretch_coord(xj[c + 1], xk[c + 1], z) - mu[c + 1];
        unsigned pk[3];
        split3_pair(v0, v1, pk);
#pragma unroll
        for (int pc = 0; pc < 3; ++pc) *reinterpret_cast<unsigned *>(row + pc * plane + c) = pk[pc];
    }
    if (lane == 0) {
        b.z[w] = z;
        b.u[w] = u;
        b.j[w] = j;
    }
}

template <bool REPLAY>
static __global__ void __launch_bounds__(256) accept_recompute_kernel(const RunParams p, const BatchBuf b, long long h, int d,
                                                               long long n, int store, long long sidx) {
    const unsigned w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const unsigned W = p.shard_end - p.shard_begin;
    if (w >= W) return;
    const unsigned i = p.shard_begin + w;
    const unsigned batch = (unsigned)(h & 1);
    const size_t k = (size_t)(batch ? p.nhalf : 0u) + i;
    const double p1 = b.p1[w], p0 = p.lp[k], z = b.z[w];
    const bool acc = accept_exact<false>(p.nm1, z, p1, p0, b.u[w]);  // :260
    double *xk = p.x + k * d;
    const double *xj = p.x + (size_t)b.j[w] * d;
    const size_t o = store ? chain_row(p, sidx, batch, i) : 0;
    if (acc || store) {
        for (int c = lane; c < d; c += 32) {
            const double xo = xk[c];
            const double v = acc ? stretch_coord(xj[c], xo, z) : xo;  // :255 again, same bits
            if (acc) xk[c] = v;                                                  // :261
            if (store) __stcs(p.chain_x + o * d + c, v);                         // :268-272
        }
    }
    if (lane == 0) {
        if (acc) {
            p.lp[k] = p1;
            p.nacc[k] += 1u;
        }
        if (batch == 1 && n == 0) {
            p.nacc[i] = 0u;
            p.nacc[(size_t)p.nhalf + i] = 0u;
        }
        if (store) __stcs(p.chain_lp + o, acc ? p1 : p0);
    }
}

// ------------------------------------------------------------------ dense Gaussian, FP64
// params (device): mu[d], A[d][d] row-major, lognorm.  A is staged transposed in shared memory
// (At[j][i], conflict-free), the centred points per warp in shared memory (broadcast reads).
// logp = lognorm - 0.5 * sum_i y_i^2;  FMA accumulation, warp-tree reduction: agrees with the
// oracle's sequential order to ~1e-14 relative (tolerance stated in the tests: 1e-12).
constexpr int kWideMaxD = 128;
constexpr int kWideThreads = 512;  // 16 warps
constexpr int kWidePts = 4;        // points per warp per pass (register tile: 4 points x 4 rows per lane)

// Register-tiled: a warp processes 4 points at once, lane l owns rows l, l+32, l+64, l+96 of y for each
// of them (16 FP64 accumulators), so every A element read from shared memory feeds 4 FMAs and every
// centred coordinate (broadcast 32-byte read of the 4 points) feeds 4 FMAs: 16 DFMA per 6 LDS -- the
// FP64 pipe, not the LSU, is the bound.  At is padded to 128 rows of zeros (no masks in the loop).
// Accumulation order per (point, row) is j = 0..d-1 with FMA, then rows in order, then the xor tree.
static __global__ void __launch_bounds__(kWideThreads, 1) gaussian_wide_logp_kernel(const double *__restrict__ X,
                                                                              double *__restrict__ out, long long npts,
                                                                              int d, const double *__restrict__ prm,
                                                                              const double *__restrict__ At_g) {
    extern __shared__ double sm[];
    double *At = sm;                          // [d][128]  At[j*128 + i] = A[i][j], zero for i >= d (At_g: same, in global)
    double *cb = sm + (size_t)d * 128;        // [warps][d][kWidePts]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    for (int e = threadIdx.x * 2; e < d * 128; e += blockDim.x * 2)  // coalesced 16-byte copies of the pre-transposed matrix
        *reinterpret_cast<double2 *>(At + e) = *reinterpret_cast<const double2 *>(At_g + e);
    __syncthreads();
    const double lognorm = prm[d + (size_t)d * d];
    double *c = cb + (size_t)wib * d * kWidePts;
    const long long ngroups = (npts + kWidePts - 1) / kWidePts;
    for (long long g = (long long)blockIdx.x * nwarp + wib; g < ngroups; g += (long long)gridDim.x * nwarp) {
        const long long pt0 = g * kWidePts;
#pragma unroll
        for (int w = 0; w < kWidePts; ++w) {
            const long long pt = pt0 + w;
            for (int j = lane; j < d; j += 32) c[j * kWidePts + w] = pt < npts ? X[pt * d + j] - prm[j] : 0.0;
        }
        __syncwarp();
        double acc[kWidePts][4];
#pragma unroll
        for (int w = 0; w < kWidePts; ++w)
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[w][r] = 0.0;
        for (int j = 0; j < d; ++j) {
            const double2 c01 = *reinterpret_cast<const double2 *>(c + j * kWidePts);
            const double2 c23 = *reinterpret_cast<const double2 *>(c + j * kWidePts + 2);
            const double cj[4] = {c01.x, c01.y, c23.x, c23.y};
            const double *row = At + j * 128 + lane;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const double a = row[32 * r];
#pragma unroll
                for (int w = 0; w < kWidePts; ++w) acc[w][r] = fma(a, cj[w], acc[w][r]);
            }
        }
#pragma unroll
        for (int w = 0; w < kWidePts; ++w) {
            double ss = 0.0;
#pragma unroll
            for (int r = 0; r < 4; ++r) ss = fma(acc[w][r], acc[w][r], ss);
            for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
            if (lane == 0 && pt0 + w < npts) out[pt0 + w] = lognorm - 0.5 * ss;
        }
        __syncwarp();
    }
}

// Dense Gaussian for 128 < d <= kHugeMaxD: the same register tile and accumulation order, in blocks of 128 rows, with the
// transposed matrix At_g[j][dpad] (dpad = d rounded up to 128, zero rows past d) read from L2 instead of shared memory
// (8 d^2 bytes no longer fit).  The reference takes any d (a user closure, src/samplers.jl:257); no tensor-core path here.
constexpr int kHugeMaxD = 4096;
static __global__ void __launch_bounds__(kWideThreads, 1) gaussian_huge_logp_kernel(const double *__restrict__ X,
                                                                                   double *__restrict__ out, long long npts,
                                                                                   int d, int dpad,
                                                                                   const double *__restrict__ prm,
                                                                                   const double *__restrict__ At_g) {
    extern __shared__ double sm[];  // [warps][d][kWidePts]: the centred points of each warp's group
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const double lognorm = prm[d + (size_t)d * d];
    double *c = sm + (size_t)wib * d * kWidePts;
    const long long ngroups = (npts + kWidePts - 1) / kWidePts;
    for (long long g = (long long)blockIdx.x * nwarp + wib; g < ngroups; g += (long long)gridDim.x * nwarp) {
        const long long pt0 = g * kWidePts;
#pragma unroll
        for (int w = 0; w < kWidePts; ++w) {
            const long long pt = pt0 + w;
            for (int j = lane; j < d; j += 32) c[j * kWidePts + w] = pt < npts ? X[pt * d + j] - prm[j] : 0.0;
        }
        __syncwarp();
        double ss[kWidePts];
#pragma unroll
        for (int w = 0; w < kWidePts; ++w) ss[w] = 0.0;
        for (int rb = 0; rb < dpad; rb += 128) {  // rows rb + lane + 32 r of y
            double acc[kWidePts][4];
#pragma unroll
            for (int w = 0; w < kWidePts; ++w)
#pragma unroll
                for (int r = 0; r < 4; ++r) acc[w][r] = 0.0;
            const double *col = At_g + rb + lane;
            for (int j = 0; j < d; ++j) {
                const double2 c01 = *reinterpret_cast<const double2 *>(c + j * kWidePts);
                const double2 c23 = *reinterpret_cast<const double2 *>(c + j * kWidePts + 2);
                const double cj[4] = {c01.x, c01.y, c23.x, c23.y};
                const double *row = col + (size_t)j * dpad;
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const double a = __ldg(row + 32 * r);
#pragma unroll
                    for (int w = 0; w < kWidePts; ++w) acc[w][r] = fma(a, cj[w], acc[w][r]);
                }
            }
#pragma unroll
            for (int w = 0; w < kWidePts; ++w)
#pragma unroll
                for (int r = 0; r < 4; ++r) ss[w] = fma(acc[w][r], acc[w][r], ss[w]);
        }
#pragma unroll
        for (int w = 0; w < kWidePts; ++w) {
            double s = ss[w];
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0 && pt0 + w < npts) out[pt0 + w] = lognorm - 0.5 * s;
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------ exponential, any d (README.md:15, d > 1: independent Exp(1))
// The dimensions without a compiled fused kernel (d = 7, 9, 11, 13-15, d > 16) take the batched half-step with this
// kernel: one thread per point, the components summed in index order with the oracle's operations -> bit-identical.
static __global__ void __launch_bounds__(256) exponential_wide_logp_kernel(const double *__restrict__ X, double *__restrict__ out,
                                                                          long long npts, int d) {
    const long long pt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (pt >= npts) return;
    const double *x = X + pt * d;
    double s = x[0];
    bool neg = x[0] < 0.0;
    for (int c = 1; c < d; ++c) {
        neg = neg || (x[c] < 0.0);
        s = dadd(s, x[c]);
    }
    out[pt] = neg ? -CUDART_INF : -s;
}

// ------------------------------------------------------------------ logistic regression, FP64
// data: X[N][d] float32 row-major then y[N] float32 (0/1); params: [prior_sigma].
//   logp(theta) = sum_n (y_n s_n - softplus(s_n)) - 0.5 |theta|^2 / sigma^2,  s_n = x_n . theta
// Exact FP64 reference path: grid (point tiles of 32) x (data chunks); a CTA keeps 32 points'
// theta in shared memory, each thread streams data rows and accumulates the 32 partial sums
// in registers; CTA tree reduction into part[chunk][point], finished in fixed chunk order
// (bit-reproducible).  Summation order differs from the oracle's sequential sum: tolerance
// 1e-10 relative on logp (stated in the tests).
constexpr int kLogitTile = 32;

__device__ __forceinline__ double softplus64(double s) { return fmax(s, 0.0) + log1p(exp(-fabs(s))); }

// part[chunk][pt] partial sums, then a fixed-order finish: bit-reproducible run to run.
static __global__ void __launch_bounds__(256) logistic_logp_kernel(const double *__restrict__ TH, double *__restrict__ part,
                                                            long long npts, int d, const float *__restrict__ X,
                                                            const float *__restrict__ yv, long long N,
                                                            long long rows_per_chunk) {
    extern __shared__ double sm[];
    double *th = sm;                                  // [kLogitTile][d]
    double *red = sm + (size_t)kLogitTile * d;        // [warps][kLogitTile]
    const long long pt0 = (long long)blockIdx.x * kLogitTile;
    const int npt = (int)min((long long)kLogitTile, npts - pt0);
    for (int e = threadIdx.x; e < kLogitTile * d; e += blockDim.x)
        th[e] = (e / d) < npt ? TH[pt0 * d + e] : 0.0;
    __syncthreads();
    double acc[kLogitTile];
#pragma unroll
    for (int w = 0; w < kLogitTile; ++w) acc[w] = 0.0;
    const long long n0 = (long long)blockIdx.y * rows_per_chunk, n1 = min(N, n0 + rows_per_chunk);
    for (long long n = n0 + threadIdx.x; n < n1; n += blockDim.x) {
        const float *xr = X + n * d;
        const double yn = (double)yv[n];
#pragma unroll
        for (int w = 0; w < kLogitTile; ++w) {
            double s = 0.0;
            for (int c = 0; c < d; ++c) s = fma((double)xr[c], th[w * d + c], s);
            acc[w] += yn * s - softplus64(s);
        }
    }
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
#pragma unroll
    for (int w = 0; w < kLogitTile; ++w) {
        double v = acc[w];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[wib * kLogitTile + w] = v;
    }
    __syncthreads();
    if (threadIdx.x < npt) {
        double v = 0.0;
        for (int k = 0; k < nwarp; ++k) v += red[k * kLogitTile + threadIdx.x];
        part[(size_t)blockIdx.y * npts + pt0 + threadIdx.x] = v;
    }
}

static __global__ void logistic_finish_kernel(const double *__restrict__ TH, const double *__restrict__ part,
                                       double *__restrict__ out, long long npts, int d, int nchunks, double inv2s2) {
    const long long pt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (pt >= npts) return;
    double v = 0.0;
    for (int k = 0; k < nchunks; ++k) v += part[(size_t)k * npts + pt];
    double nn = 0.0;
    for (int c = 0; c < d; ++c) nn = fma(TH[pt * d + c], TH[pt * d + c], nn);
    out[pt] = v - nn * inv2s2;
}

}  // namespace kmc
