// kmc_device.cuh -- device-side building blocks of the emcee stretch-move kernels (sm_100a).
//
// Arithmetic contract (shared with oracle/kmc_oracle.c): IEEE binary64, round-to-nearest and
// NO fused multiply-add on anything that decides accept/reject or produces chain state.  The
// reference is Julia, which never contracts a*b+c (src/samplers.jl:255,:260), so every such
// operation goes through the __d*_rn intrinsics, which nvcc never fuses.
#pragma once
#include <cstdint>
#ifndef KMC_U48_BITS
#define KMC_U48_BITS 0
#endif
#include <cuda_runtime.h>

namespace kmc {

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }

// One coordinate of the stretch proposal y = xj + z (xk - xj) (src/samplers.jl:255): every kernel that forms or
// recomputes a proposal uses this one spelling, so they all produce the same bits.
__device__ __forceinline__ double stretch_coord(double xj, double xk, double z) { return dadd(xj, dmul(z, dsub(xk, xj))); }

// The reference's thinning clock (src/samplers.jl:245, :268): its loop variable n = t + 1 - nburnin (0 at the last
// burn-in iteration), rem(n, nthin) and the number of samples stored before n.  Phase is the type the phase is kept
// in (a kernel may keep it in 32 bits).
template <class Phase = long long>
struct ThinClock {
    long long n;
    Phase phase;
    long long sidx;
    // the clock at 0-based iteration t
    __host__ __device__ static ThinClock at(long long t, long long nburnin, long long nthin) {
        const long long n = t + 1 - nburnin;
        long long ph = n % nthin;  // floored: n < 0 during burn-in
        if (ph < 0) ph += nthin;
        return ThinClock{n, (Phase)ph, n >= 1 ? (n - 1) / nthin : 0};
    }
    __host__ __device__ bool store() const { return n > 0 && phase == 0; }  // :268  n>0 && rem(n,nthin)==0
    __host__ __device__ bool burnin_end() const { return n == 0; }          // :285-288 accept counters restart
    // to the next iteration; `stored` is store() of this one
    __host__ __device__ void advance(bool stored, Phase nthin) {
        if (stored) ++sidx;
        ++n;
        if (++phase == nthin) phase = 0;
    }
};

// ------------------------------------------------------------------ FP64 -> three bf16 pieces (tcgen05 operands)
// Walker coordinates for the tensor-core log-densities: v is rounded ONCE to FP32 (24 significant
// bits) and that value is split exactly: h0 = RN_bf16(f), r1 = f - h0, h1 = RN_bf16(r1),
// r2 = r1 - h1, h2 = RN_bf16(r2) = r2.  Both subtractions are exact in FP32 (the residual of
// rounding a 24-bit number to 8 bits has at most 16 significant bits, then 8), so
// h0 + h1 + h2 == RN_f32(v).  Two coordinates at a time: one F2F.F32.F64 each, then per piece one
// packed F2FP.BF16 + two integer unpacks + two FSUB -- a direct FP64 split costs four XU-pipe
// F2F conversions per coordinate and piece and was the bound of the fused kernel's proposal phase.
// pk[pc] = bf16(v0 piece) | bf16(v1 piece) << 16.  Every kernel that feeds points to a tcgen05
// Gaussian GEMM uses this one function, so their operands agree bit for bit.
__device__ __forceinline__ void split3_pair(double v0, double v1, unsigned (&pk)[3]) {
    float f0 = __double2float_rn(v0), f1 = __double2float_rn(v1);
#pragma unroll
    for (int pc = 0; pc < 3; ++pc) {
        unsigned u;
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(u) : "f"(f1), "f"(f0));  // upper half <- f1, lower half <- f0
        pk[pc] = u;
        if (pc < 2) {
            f0 = __fsub_rn(f0, __uint_as_float(u << 16));
            f1 = __fsub_rn(f1, __uint_as_float(u & 0xFFFF0000u));
        }
    }
}

// ------------------------------------------------------------------ Philox4x32-10
struct Philox4 {
    uint32_t r0, r1, r2, r3;
};

// Round keys k + r*W for r = 0..9, precomputed on the host and passed in the kernel arguments
// (constant bank), so a round is exactly 2 IMAD.WIDE + 2 three-input LOP3.
struct PhiloxKeys {
    uint32_t k0[10], k1[10];
};

__host__ __device__ inline PhiloxKeys philox_keys(uint64_t seed) {
    PhiloxKeys ks;
    uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) {
        ks.k0[r] = a;
        ks.k1[r] = b;
        a += 0x9E3779B9u;
        b += 0xBB67AE85u;
    }
    return ks;
}

__device__ __forceinline__ void mul_wide(uint32_t a, uint32_t b, uint32_t &hi, uint32_t &lo) {
    asm("{\n\t.reg .u64 t;\n\tmul.wide.u32 t, %2, %3;\n\tmov.b64 {%1, %0}, t;\n\t}" : "=r"(hi), "=r"(lo) : "r"(a), "r"(b));
}

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 const PhiloxKeys &ks) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        mul_wide(0xD2511F53u, c0, hi0, lo0);
        mul_wide(0xCD9E8D57u, c2, hi1, lo1);
        c0 = hi1 ^ c1 ^ ks.k0[r];
        c1 = lo1;
        c2 = hi0 ^ c3 ^ ks.k1[r];
        c3 = lo0;
    }
    return Philox4{c0, c1, c2, c3};
}

__device__ __forceinline__ uint32_t lemire_retry(const PhiloxKeys &ks, uint32_t walker, uint32_t iter_lo,
                                              uint32_t iter_hi, uint32_t batch, uint32_t nhalf, uint32_t lemire_t) {
    uint32_t hi, lo, attempt = 0;
    do {
        ++attempt;
        const Philox4 rr = philox4x32_10(walker, iter_lo, iter_hi, batch | (attempt << 8), ks);
        mul_wide(rr.r0, nhalf, hi, lo);
    } while (lo < lemire_t);
    return hi;
}

// One walker-step's draws, in the reference's order: partner (src/samplers.jl:250), the
// uniform behind z (:252 -> :230), the accept uniform (:260).  counter = (walker id,
// iteration lo, iteration hi, batch | attempt<<8), key = seed.  The partner uses Lemire's
// multiply-shift with rejection, so it is exactly uniform on [0, nhalf) like rand(range).
__device__ __forceinline__ void draw(const PhiloxKeys &ks, uint32_t walker, uint32_t iter_lo, uint32_t iter_hi,
                                     uint32_t batch, uint32_t nhalf, uint32_t lemire_t, uint32_t &partner_local,
                                     double &uz, double &uacc) {
    const Philox4 r = philox4x32_10(walker, iter_lo, iter_hi, batch, ks);
    uint32_t hi, lo;
    mul_wide(r.r0, nhalf, hi, lo);
    if (lo < lemire_t)  // probability < nhalf / 2^32 per draw: kept out of line
        hi = lemire_retry(ks, walker, iter_lo, iter_hi, batch, nhalf, lemire_t);
    partner_local = hi;
    const uint64_t bz = ((uint64_t)r.r1 << 16) | (r.r2 >> 16);
    const uint64_t ba = ((uint64_t)(r.r2 & 0xFFFFu) << 32) | r.r3;
#if KMC_U48_BITS
    // the same values without the two U64 -> F64 conversions (XU pipe): 1 + b*2^-48 assembled in the mantissa, then an
    // exact subtraction of 1
    uz = __dadd_rn(__longlong_as_double((long long)(0x3FF0000000000000ULL | (bz << 4))), -1.0);
    uacc = __dadd_rn(__longlong_as_double((long long)(0x3FF0000000000000ULL | (ba << 4))), -1.0);
#else
    uz = (double)bz * 0x1p-48;    // exact: 48-bit integer times a power of two
    uacc = (double)ba * 0x1p-48;
#endif
}

// Two counter-based standard normals from one Philox block: words r0, r1 -> uniforms in (0, 1] and [0, 1) ->
// Box-Muller.  c3 carries the stream tag that keeps the users of this helper apart (make_theta0s: 0x4D54 << 16,
// metropolis: 0x4D48 << 16 | pair); the block is returned so that a caller can use r2 and r3 too.
__device__ __forceinline__ Philox4 philox_normals(const PhiloxKeys &ks, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                  double &z0, double &z1) {
    const Philox4 r = philox4x32_10(c0, c1, c2, c3, ks);
    const double u1 = ((double)r.r0 + 1.0) * 0x1p-32;  // (0, 1]
    const double u2 = (double)r.r1 * 0x1p-32;          // [0, 1)
    const double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    z0 = rad * cs;
    z1 = rad * sn;
    return r;
}

// ------------------------------------------------------------------ log-density plugins
// Each plugin is a POD passed BY VALUE in the kernel arguments, so its parameters sit in the
// constant bank and feed the FP64 pipe directly (no loads).  logpdf() follows the operation
// order written in oracle/kmc_oracle.c::kmo_logpdf exactly.

constexpr int KIND_EXPONENTIAL = 0;
constexpr int KIND_ROSENBROCK = 1;
constexpr int KIND_GAUSSIAN = 2;
constexpr int KIND_LOGNORMAL = 3;
constexpr int KIND_LOGISTIC = 4;

// README.md:15  logpdf(x) = x<0 ? -Inf : -x   (d>1: independent Exp(1) components)
template <int D>
struct Exponential {
    static constexpr int kind = KIND_EXPONENTIAL;
    static constexpr int nparams = 0;
    double unused;
    __device__ __forceinline__ double logpdf(const double (&x)[D]) const {
        double s = x[0];
        bool neg = x[0] < 0.0;
#pragma unroll
        for (int c = 1; c < D; ++c) {
            neg = neg || (x[c] < 0.0);
            s = dadd(s, x[c]);
        }
        return neg ? -CUDART_INF : -s;
    }
};

// Correctly rounded a/b from the correctly rounded reciprocal y = RN(1/b) (computed on the
// host): two Markstein corrections, q <- q + (a - b*q)*y with exact FMA residuals.  After the
// first correction q is a faithful quotient, so the second returns RN(a/b) (Markstein 1990;
// Muller et al., Handbook of Floating-Point Arithmetic, thm 5.4) -- the same bits as
// __ddiv_rn / the oracle's `/`, in 5 FP64 instructions instead of ~20.  Valid away from
// overflow/underflow; anything else (and y == 0, set by the host when b is out of range)
// takes __ddiv_rn.
__device__ __forceinline__ double ddiv_by(double a, double b, double y) {
    const double aa = fabs(a);
    if (y != 0.0 && aa > 0x1p-900 && aa < 0x1p900) {
        const double q0 = a * y;
        const double r0 = fma(-b, q0, a);
        const double q1 = fma(r0, y, q0);
        const double r1 = fma(-b, q1, a);
        return fma(r1, y, q1);
    }
    return __ddiv_rn(a, b);
}

// test/runtests.jl:68  -(100*(x2 - x1^2)^2 + (1 - x1)^2)/20, params [a, b, T] (+ RN(1/T), host-filled)
template <int D>
struct Rosenbrock {
    static_assert(D == 2, "rosenbrock is 2-D");
    static constexpr int kind = KIND_ROSENBROCK;
    static constexpr int nparams = 3;
    double p[4];
    __device__ __forceinline__ double logpdf(const double (&x)[D]) const {
        const double t = dsub(x[1], dmul(x[0], x[0]));
        const double q = dmul(p[1], dmul(t, t));
        const double m = dsub(p[0], x[0]);
        const double r = dadd(q, dmul(m, m));
        return ddiv_by(-r, p[2], p[3]);
    }
};

// test/runtests.jl:53,61  params [mu(D), A(D*D row-major), lognorm]
template <int D>
struct Gaussian {
    static constexpr int kind = KIND_GAUSSIAN;
    static constexpr int nparams = D + D * D + 1;
    double p[D + D * D + 1];
    __device__ __forceinline__ double logpdf(const double (&x)[D]) const {
        double c[D];
#pragma unroll
        for (int j = 0; j < D; ++j) c[j] = dsub(x[j], p[j]);
        double ss = 0.0;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            double y = 0.0;
#pragma unroll
            for (int j = 0; j < D; ++j) y = dadd(y, dmul(p[D + i * D + j], c[j]));
            ss = dadd(ss, dmul(y, y));
        }
        return dsub(p[D + D * D], dmul(0.5, ss));
    }
};

// test/runtests.jl:56  LogNormal(mu, sigma); params [mu, sigma, log(sigma)+0.5*log(2pi)]
template <int D>
struct LogNormal {
    static_assert(D == 1, "lognormal is 1-D");
    static constexpr int kind = KIND_LOGNORMAL;
    static constexpr int nparams = 3;
    double p[3];
    __device__ __forceinline__ double logpdf(const double (&x)[D]) const {
        if (!(x[0] > 0.0)) return (x[0] != x[0]) ? x[0] : -CUDART_INF;
        const double lx = log(x[0]);
        const double t = ddiv(dsub(lx, p[0]), p[1]);
        return dsub(dsub(-lx, dmul(0.5, dmul(t, t))), p[2]);
    }
};

// ------------------------------------------------------------------ row access
// Walker rows are contiguous ([nw][D] row-major): a partner gather touches ceil(8D/32)
// sectors instead of D sectors with a component-major layout, and for even D the active
// walker's own row is a coalesced 128-bit access.
template <int D>
__device__ __forceinline__ void load_row(const double *__restrict__ p, double (&v)[D]) {
    if constexpr (D % 2 == 0) {
#pragma unroll
        for (int c = 0; c < D; c += 2) {
            const double2 t = *reinterpret_cast<const double2 *>(p + c);
            v[c] = t.x;
            v[c + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int c = 0; c < D; ++c) v[c] = p[c];
    }
}

// L2-coherent gather (ld.global.cg): partner rows are written by other SMs between
// half-steps of the persistent kernel, so they must not be served from a stale L1 line.
template <int D>
__device__ __forceinline__ void load_row_cg(const double *p, double (&v)[D]) {
    if constexpr (D % 2 == 0) {
#pragma unroll
        for (int c = 0; c < D; c += 2) {
            const double2 t = __ldcg(reinterpret_cast<const double2 *>(p + c));
            v[c] = t.x;
            v[c + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int c = 0; c < D; ++c) v[c] = __ldcg(p + c);
    }
}

template <int D>
__device__ __forceinline__ void store_row(double *p, const double (&v)[D]) {
    if constexpr (D % 2 == 0) {
#pragma unroll
        for (int c = 0; c < D; c += 2) *reinterpret_cast<double2 *>(p + c) = make_double2(v[c], v[c + 1]);
    } else {
#pragma unroll
        for (int c = 0; c < D; ++c) p[c] = v[c];
    }
}

// Streaming store for the chain (written once, never re-read by the sampler).
template <int D>
__device__ __forceinline__ void store_row_cs(double *p, const double (&v)[D]) {
    if constexpr (D % 2 == 0) {
#pragma unroll
        for (int c = 0; c < D; c += 2) __stcs(reinterpret_cast<double2 *>(p + c), make_double2(v[c], v[c + 1]));
    } else {
#pragma unroll
        for (int c = 0; c < D; ++c) __stcs(p + c, v[c]);
    }
}

}  // namespace kmc
