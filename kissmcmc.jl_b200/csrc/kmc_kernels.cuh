// kmc_kernels.cuh -- the fused stretch-move kernels (thread-per-walker family, FP64).
//
// One walker-step fuses everything inside the reference's threaded loop body,
// src/samplers.jl:249-272: partner draw, z draw, proposal, log-density, accept test,
// in-place update, accept counter, thinned chain store.
//
// emcee_run_kernel advances a RANGE of half-steps in ONE launch.  Every CTA owns a fixed,
// contiguous slice of walker positions of BOTH halves for the whole launch, and consecutive
// half-steps are separated by a grid-wide barrier (the reference's thread join at the end of
// each `Threads.@threads` sweep, :248/:273).  Two residency modes for the owned state:
//   SMEM=true   x / logp / accept counters of the CTA's walkers live in shared memory for the
//               whole launch (component-major, conflict-free); global x is only written on
//               accept (so partners can gather it) and logp / counters are written back once
//               at the end.  Used when the ensemble fits the SMs' aggregate shared memory
//               (2^20 2-D walkers: 28 B x 7086 walkers = 194 KB per SM).
//   SMEM=false  state stays in L2/HBM; any ensemble size.
// With a range of one half-step the kernel degenerates to "one launch per half-step".
#pragma once
#include <math_constants.h>
#include <type_traits>

#include "kmc_device.cuh"

namespace kmc {

// Launch shape of emcee_run_kernel.  Small rows: 2 CTAs x <=448 threads per SM in <= 72
// registers, 4 walkers in flight per thread; wider rows (more live FP64 values per walker):
// 1 CTA x <=256 threads with up to 255 registers, 1-2 walkers in flight.
template <int D>
__host__ __device__ constexpr int max_threads() { return D <= 4 ? 448 : 256; }
template <int D>
__host__ __device__ constexpr int min_blocks() { return D <= 4 ? 2 : 1; }
template <int D>
__host__ __device__ constexpr int in_flight() { return D <= 2 ? 2 : (D <= 8 ? 2 : 1); }

struct RunParams {
    double *x;          // [nw][D] row-major walker positions (theta0s, :198)
    double *lp;         // [nw] current log-density (p0s, :209)
    unsigned *nacc;     // [nw] accept counters (naccept, :242)
    double *chain_x;    // [ns][nw][D] sample-major thinned chain (coalesced stores)
    double *chain_lp;   // [ns][nw]
    const long long *rp_partner;  // replay draws, indexed ((t-rp_t0)*2+batch)*nhalf + i
    const double *rp_z;
    const double *rp_u;
    long long rp_t0;
    long long nw;
    unsigned nhalf;
    unsigned per_cta;   // walker positions (of each half) owned by one CTA
    unsigned shard_begin, shard_end;  // positions of each half this sampler updates (whole half: 0, nhalf)
    long long chain_nw;               // walkers in the chain store: 2*(shard_end-shard_begin)
    long long h0, h1;   // half-step range, h = 2*t + batch, t = 0-based outer iteration
    long long n0;       // the reference's loop variable n (:245) at t = h0/2
    long long phase0;   // n0 mod nthin (floored)
    long long sidx0;    // samples already stored before n0
    long long nthin, ns;
    double sia, span, nm1;  // sqrt(1/a), sqrt(a)-sqrt(1/a), (N-1)
    float nm1f, margin;     // fast accept filter: (N-1) and its rigorous error margin
    PhiloxKeys keys;        // Philox round keys of the seed
    unsigned id_base[2];    // Philox walker id = id_base[batch] + i (low 32 bits of the global walker index)
    unsigned lemire_t;      // (2^32 - nhalf) mod nhalf
    unsigned long long *barrier;  // grid barrier arrival counter (monotonic)
    unsigned long long bar_base;  // its value when this launch starts
    // peer mode (one ensemble sharded over GPUs): partner rows are gathered straight from the
    // owner GPU's memory over NVLink and ranks meet at a system-scope flag barrier per half-step
    const double *peer_x[8];          // x of every rank (own rank: the local pointer)
    unsigned long long *peer_flags[8];  // flag array [npeers] of every rank
    int npeers, rank;
    unsigned long long epoch_base;    // cross-GPU barrier epochs completed before this launch
};

// ------------------------------------------------------------------ grid barrier
// Monotonic arrival counter; cooperative launch guarantees all CTAs are resident.
// arrive: all threads' stores -> bar.sync -> thread 0: red.release.gpu (+1)
// wait:   thread 0 polls (relaxed), then fence.acq_rel.gpu once -> bar.sync -> everyone
//         gathers partner rows with ld.global.cg (L2), never from L1.
// The two halves are split so that work that does not depend on other CTAs (the next
// half-step's Philox draws) runs between arrive and wait.
__device__ __forceinline__ void barrier_arrive(unsigned long long *ctr) {
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(ctr) : "memory");
}
__device__ __forceinline__ void barrier_wait(const unsigned long long *ctr, unsigned long long target) {
    unsigned long long v;
    long long t0 = 0;
    unsigned spins = 0;
    do {
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(ctr) : "memory");
        if (v < target && (++spins & 0xFFFu) == 0) {  // watchdog (~20 s): a lost CTA must not hang the device
            if (t0 == 0) t0 = clock64();
            else if (clock64() - t0 > 40000000000LL) __trap();
        }
    } while (v < target);
    asm volatile("fence.acq_rel.gpu;" ::: "memory");
}

// The shared-memory kernel's wait: acquire loads (LDG.STRONG.GPU + CCTL.IVALL) instead of relaxed loads + fence.acq_rel.gpu
// (MEMBAR.ALL.GPU + ERRBAR): measured 0.4 us per half-step of that kernel.  Every poll invalidates the SM's L1, which that
// kernel never uses for global data (partner rows are .cg loads).
__device__ __forceinline__ void barrier_wait_acquire(const unsigned long long *ctr, unsigned long long target) {
    unsigned long long v;
    long long t0 = 0;
    unsigned spins = 0;
    do {
        asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(ctr) : "memory");
        if (v < target && (++spins & 0xFFFu) == 0) {  // watchdog (~20 s)
            if (t0 == 0) t0 = clock64();
            else if (clock64() - t0 > 40000000000LL) __trap();
        }
    } while (v < target);
}

// The join between two half-steps of a persistent kernel (the reference's join after each sweep, :248/:273), local to
// this GPU.  The CTA's stores are done before thread 0 arrives; shadow() is work independent of the other CTAs, run
// between arrive and wait (without it thread 0 arrives and waits at once).  The barrier is polled by thread 0 with
// relaxed loads and one fence, or, with LAST_WARP_ACQUIRE, by the last warp with acquire loads (thread 0's warp is
// still behind its release).
struct NoShadow {
    __device__ void operator()() const {}
};
template <bool LAST_WARP_ACQUIRE = false, class Shadow = NoShadow>
__device__ __forceinline__ void grid_join(const RunParams &p, unsigned long long &target, Shadow shadow = {}) {
    auto arrive = [&] { barrier_arrive(p.barrier); };
    auto wait = [&] {
        if constexpr (LAST_WARP_ACQUIRE) {
            if (threadIdx.x == blockDim.x - 32) barrier_wait_acquire(p.barrier, target);
        } else {
            if (threadIdx.x == 0) barrier_wait(p.barrier, target);
        }
    };
    target += gridDim.x;
    __syncthreads();
    if constexpr (std::is_same<Shadow, NoShadow>::value) {
        static_assert(!LAST_WARP_ACQUIRE, "without shadow work thread 0 arrives and polls");
        if (gridDim.x > 1) {
            if (threadIdx.x == 0) {
                arrive();
                wait();
            }
            __syncthreads();
        }
    } else {
        if (gridDim.x > 1 && threadIdx.x == 0) arrive();
        shadow();
        if (gridDim.x > 1) {
            wait();
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------ accept test
// Decides  ((N-1)*log(z) + p1) - p0 >= log(u)   (src/samplers.jl:260).
// Fast filter: t = (p1-p0) + ln2*q,  q = (N-1)*lg2f(z) - lg2f(u)  with FP32 MUFU logs.  The
// error of t is bounded by `margin` (set by the host: (N-1+64)*2e-6, >3x the worst case of
// two MUFU.LG2 errors (2^-22.6 absolute on the mantissa part + one FP32 rounding of the
// result), two FP64->FP32 input roundings and one FP32 fma, for |lg2 z| <= 4 and
// |lg2 u| <= 100), so |t| > margin decides exactly like the FP64 expression.  Anything closer,
// non-finite or outside that range (q = NaN) takes the exact FP64 path: the decisions are
// those of the exact expression, bit for bit.
template <bool SKIP_LOGZ>
__device__ __forceinline__ bool accept_exact(double nm1, double z, double p1, double p0, double u) {
    double lhs;
    if constexpr (SKIP_LOGZ) lhs = dsub(p1, p0);  // (N-1)*log(z) == 0 exactly: N == 1 and z finite positive
    else lhs = dsub(dadd(dmul(nm1, log(z)), p1), p0);
    return lhs >= log(u);
}

__device__ __forceinline__ float lg2_approx(float v) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}

template <bool REPLAY>
__device__ __forceinline__ float filter_q(const RunParams &p, double z, double u) {
    const float zf = (float)z, uf = (float)u;
    bool ok = uf > 1e-30f;  // false for NaN
    if constexpr (REPLAY) ok = ok && uf < 1e30f;                  // Philox: u < 1 always
    ok = ok && zf > 0.0625f && zf < 16.0f;
    const float q = fmaf(p.nm1f, lg2_approx(zf), -lg2_approx(uf));
    return ok ? q : CUDART_NAN_F;
}

// ------------------------------------------------------------------ draws for one walker-step
template <bool REPLAY>
__device__ __forceinline__ void step_draws(const RunParams &p, long long h, unsigned i, unsigned &j, double &z,
                                           double &u) {
    if constexpr (REPLAY) {
        const long long slot = (h - 2 * p.rp_t0) * (long long)p.nhalf + i;
        j = (unsigned)__ldcs(p.rp_partner + slot);  // global 0-based index
        z = __ldcs(p.rp_z + slot);
        u = __ldcs(p.rp_u + slot);
    } else {
        const unsigned long long t = (unsigned long long)(h >> 1);
        const unsigned batch = (unsigned)(h & 1);
        unsigned pl;
        double uz;
        draw(p.keys, p.id_base[batch] + i, (unsigned)t, (unsigned)(t >> 32), batch, p.nhalf, p.lemire_t, pl, uz, u);
        j = (batch ? 0u : p.nhalf) + pl;                 // :247 passive half
        const double s = dadd(dmul(uz, p.span), p.sia);  // :227
        z = dmul(s, s);
    }
}

// The rare exact accept path: re-derive the accept uniform and evaluate the FP64 expression.
template <bool REPLAY, bool SKIP_LOGZ>
__device__ __forceinline__ bool accept_slow(const RunParams &p, long long h, unsigned i, double z, double p1, double p0) {
    unsigned j;
    double z2, u;
    step_draws<REPLAY>(p, h, i, j, z2, u);
    return accept_exact<SKIP_LOGZ>(p.nm1, z, p1, p0, u);
}

struct DrawRec {  // what a walker-step needs from its draws: 4 registers
    unsigned j;   // partner (global index)
    float q;      // accept-filter term, NaN = take the exact path
    double z;
};

// Row of global walker k (position i of its half) in the chain store: local shard order.
__device__ __forceinline__ size_t chain_row(const RunParams &p, long long sidx, unsigned batch, unsigned i) {
    return (size_t)sidx * p.chain_nw + (batch ? (size_t)(p.shard_end - p.shard_begin) : 0) + (i - p.shard_begin);
}

// Thinned chain store of one walker (:268-272): its current state right after its own update.
template <int D>
__device__ __forceinline__ void chain_store(const RunParams &p, size_t o, bool acc, const double (&y)[D],
                                            const double (&xk)[D], double p1, double lpk) {
    if (acc) store_row_cs<D>(p.chain_x + o * D, y);
    else store_row_cs<D>(p.chain_x + o * D, xk);
    __stcs(p.chain_lp + o, acc ? p1 : lpk);
}

// ------------------------------------------------------------------ cross-GPU pieces (peer mode)
// Partner rows that may live on another GPU: system-scope relaxed loads, never from L1.
template <int D>
__device__ __forceinline__ void load_row_sys(const double *p, double (&v)[D]) {
    if constexpr (D % 2 == 0) {
#pragma unroll
        for (int c = 0; c < D; c += 2)
            asm volatile("ld.relaxed.sys.global.v2.f64 {%0, %1}, [%2];" : "=d"(v[c]), "=d"(v[c + 1]) : "l"(p + c) : "memory");
    } else {
#pragma unroll
        for (int c = 0; c < D; ++c) asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v[c]) : "l"(p + c) : "memory");
    }
}

// One bulk (TMA) copy of a whole partner row, global/peer -> shared: a single D*8-byte request on
// the wire instead of D/2 16-byte loads; completion is counted on a CTA mbarrier.
__device__ __forceinline__ void bulk_row_g2s(void *smem_dst, const void *gsrc, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (unsigned)__cvta_generic_to_shared(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
                 : "memory");
}
__device__ __forceinline__ void kbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void kbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void kbar_wait(unsigned long long *bar, unsigned parity) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    const long long t0 = clock64();
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
        if (!done && clock64() - t0 > 20000000000LL) __trap();
    }
}

// Called by ONE CTA between two local grid barriers: publish "this GPU finished epoch e" into
// every rank's flag array (st.release.sys after the local barrier made all CTAs' writes visible
// to this thread: cumulativity carries them system-wide), then wait for every rank's flag.
__device__ __forceinline__ void cross_gpu_barrier(const RunParams &p, unsigned long long epoch) {
    if ((int)threadIdx.x < p.npeers) {
        unsigned long long *dst = p.peer_flags[threadIdx.x] + p.rank;
        asm volatile("fence.acq_rel.sys;" ::: "memory");
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(epoch) : "memory");
        const unsigned long long *mine = p.peer_flags[p.rank] + threadIdx.x;
        const long long t0 = clock64();
        unsigned long long v;
        do {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(mine) : "memory");
            if (v < epoch && clock64() - t0 > 20000000000LL) __trap();  // ~10 s watchdog: a missing peer must not hang the GPU
        } while (v < epoch);
    }
}

// Peer mode, after the local join of half-step h: every GPU has finished the half-step before anyone gathers from it.
__device__ __forceinline__ void peer_join(const RunParams &p, unsigned long long &target, long long h) {
    if (blockIdx.x == 0) cross_gpu_barrier(p, p.epoch_base + (unsigned long long)(h - p.h0) + 1);
    grid_join(p, target);
}

// ------------------------------------------------------------------ general kernel
// Owned state stays in L2/HBM; any ensemble size.  U walkers in flight per thread.
template <template <int> class Dn, int D, bool REPLAY, bool PEER = false>
static __global__ void __launch_bounds__(max_threads<D>(), min_blocks<D>()) emcee_run_kernel(const RunParams p,
                                                                                    const Dn<D> dn) {
    constexpr int U = in_flight<D>();
    const unsigned shard_size = p.shard_end - p.shard_begin;
    // peer mode: partner rows land in shared memory through bulk copies (rows of 16-byte multiples)
    constexpr bool BULK = PEER && (D % 2 == 0);
    __shared__ __align__(16) double prow[BULK ? U * max_threads<D>() * D : 1];
    __shared__ unsigned long long pbar;
    unsigned pphase = 0;
    if constexpr (BULK) {
        if (threadIdx.x == 0) kbar_init(&pbar, 1);
        __syncthreads();
    }
    const unsigned tid = threadIdx.x, nthr = blockDim.x;
    const unsigned base = p.shard_begin + blockIdx.x * p.per_cta;  // first owned position (in each half)
    const unsigned cnt = base >= p.shard_end ? 0u : min(p.per_cta, p.shard_end - base);

    DrawRec dr[U];
    auto make_draws = [&](long long h, unsigned l, DrawRec &r) {
        unsigned j;
        double z, u;
        step_draws<REPLAY>(p, h, base + l, j, z, u);  // :250, :252, (:260 uniform)
        r.j = j;
        r.z = z;
        r.q = filter_q<REPLAY>(p, z, u);
    };
#pragma unroll
    for (int q = 0; q < U; ++q) {
        const unsigned l = tid + q * nthr;
        if (l < cnt) make_draws(p.h0, l, dr[q]);
    }

    ThinClock<> clk{p.n0, p.phase0, p.sidx0};
    unsigned long long target = p.bar_base;
    for (long long h = p.h0; h < p.h1; ++h) {
        const int batch = (int)(h & 1);
        const bool store = clk.store();
        const unsigned a0 = batch ? p.nhalf : 0u;    // :247 active half

        for (unsigned g = 0; g * nthr < cnt; g += U) {  // groups of U walkers in flight
            if (g > 0) {
#pragma unroll
                for (int q = 0; q < U; ++q) {
                    const unsigned l = tid + (g + q) * nthr;
                    if (l < cnt) make_draws(h, l, dr[q]);
                }
            }
            double xj[U][D], xk[U][D], lpk[U];
            if constexpr (BULK) {  // bytes this CTA's bulk copies of the group will deliver
                if (tid == 0) {
                    unsigned rows = 0;
#pragma unroll
                    for (int q = 0; q < U; ++q) {
                        const unsigned first = (g + q) * nthr;
                        rows += first < cnt ? min(nthr, cnt - first) : 0u;
                    }
                    kbar_expect_tx(&pbar, rows * D * 8);
                }
            }
#pragma unroll
            for (int q = 0; q < U; ++q) {  // all gathers and owned rows of the group in flight together
                const unsigned l = tid + (g + q) * nthr;
                if (l < cnt) {
                    const size_t k = (size_t)a0 + base + l;
                    if constexpr (PEER) {  // the partner's owner: position inside its half / shard size
                        const unsigned pos = dr[q].j >= p.nhalf ? dr[q].j - p.nhalf : dr[q].j;
                        const double *src = p.peer_x[pos / shard_size] + (size_t)dr[q].j * D;
                        if constexpr (BULK) bulk_row_g2s(prow + ((size_t)q * nthr + tid) * D, src, D * 8, &pbar);
                        else load_row_sys<D>(src, xj[q]);
                    } else {
                        load_row_cg<D>(p.x + (size_t)dr[q].j * D, xj[q]);
                    }
                    load_row<D>(p.x + k * D, xk[q]);
                    lpk[q] = p.lp[k];
                }
            }
            if constexpr (BULK) {
                kbar_wait(&pbar, pphase);
                pphase ^= 1;
#pragma unroll
                for (int q = 0; q < U; ++q) {
                    const unsigned l = tid + (g + q) * nthr;
                    if (l < cnt) {
#pragma unroll
                        for (int c = 0; c < D; ++c) xj[q][c] = prow[((size_t)q * nthr + tid) * D + c];
                    }
                }
                __syncthreads();  // the row buffers are reused by the next group's bulk copies
            }
#pragma unroll
            for (int q = 0; q < U; ++q) {
                const unsigned l = tid + (g + q) * nthr;
                if (l >= cnt) continue;
                const size_t k = (size_t)a0 + base + l;
                const double z = dr[q].z;
                double y[D];
#pragma unroll
                for (int c = 0; c < D; ++c) y[c] = stretch_coord(xj[q][c], xk[q][c], z);  // :255
                const double p1 = dn.logpdf(y);                                            // :257
                const double tt = (p1 - lpk[q]) + (double)dr[q].q * 0.6931471805599453;  // :260
                bool acc;
                if (tt > (double)p.margin) acc = true;
                else if (tt < -(double)p.margin) acc = false;
                else acc = accept_slow<REPLAY, (D == 1 && !REPLAY)>(p, h, base + l, z, p1, lpk[q]);
                if (acc) {  // :261-265
                    store_row<D>(p.x + k * D, y);
                    p.lp[k] = p1;
                    p.nacc[k] += 1u;
                }
                if (store) chain_store<D>(p, chain_row(p, clk.sidx, (unsigned)batch, base + l), acc, y, xk[q], p1, lpk[q]);
            }
        }
        if (batch == 1) {
            if (clk.burnin_end()) {  // :285-288 burn-in counters are discarded
                for (unsigned l = tid; l < cnt; l += nthr) {
                    p.nacc[base + l] = 0u;
                    p.nacc[(size_t)p.nhalf + base + l] = 0u;
                }
            }
            clk.advance(store, p.nthin);
        }
        if (h + 1 < p.h1) {
            grid_join(p, target, [&] {
#pragma unroll
                for (int q = 0; q < U; ++q) {  // next half-step's first group of draws, in the barrier's shadow
                    const unsigned l = tid + q * nthr;
                    if (l < cnt) make_draws(h + 1, l, dr[q]);
                }
            });
            if constexpr (PEER) peer_join(p, target, h);
        }
    }
}

// ------------------------------------------------------------------ bulk (TMA) general kernel
// For HBM-resident ensembles with rows of 16-byte multiples (D even, D >= 6): every row moves as a
// bulk async copy instead of D/2 16-byte loads per thread, which cuts the number of memory requests
// per walker-step ~5x at d = 10 (the per-thread version is request/latency bound: DRAM at 42 %):
//   * the CTA's own rows of a group are ONE contiguous bulk load (global -> smem) and, after the
//     update, ONE contiguous bulk store (smem -> global): full lines, no partial-sector writes;
//     rows that were not accepted are rewritten with their old value (nobody reads the active
//     half during its own half-step);
//   * each thread gathers its partner row with one bulk request (from the owner GPU in peer mode).
// Own-row buffers are double-buffered so the store of group g overlaps the loads of group g+1.
constexpr int kBulkThreads = 256;
// KMC_BULK_STORE_ALL = 1: the CTA's own rows go back as ONE bulk store per group (rows that were not accepted are
// rewritten with their old value).  0 (default): only ACCEPTED rows are written, straight from registers -- the kernel is
// bound by its DRAM traffic and at the ~30 % acceptance of the 10-D Gaussian that removes ~50 of 368 bytes per walker-step
// (the partially covered sector at a row's end merges in L2 with the line the group's own-row load has just brought in).
#ifndef KMC_BULK_STORE_ALL
#define KMC_BULK_STORE_ALL 0
#endif
#ifndef KMC_BULK_CTAS
#define KMC_BULK_CTAS 3
#endif

__device__ __forceinline__ void bulk_s2g(void *gdst, const void *smem_src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
                 "r"((unsigned)__cvta_generic_to_shared(smem_src)), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}

template <template <int> class Dn, int D, bool PEER>
static __global__ void __launch_bounds__(kBulkThreads, KMC_BULK_CTAS) emcee_bulk_kernel(const RunParams p, const Dn<D> dn) {
    static_assert(D % 2 == 0, "rows must be multiples of 16 bytes");
    extern __shared__ __align__(128) unsigned char bulk_smem[];
    constexpr unsigned T = kBulkThreads, ROWB = D * 8;
    double *xown = reinterpret_cast<double *>(bulk_smem);                    // [2][T][D]
    double *xpart = xown + 2 * T * D;                                        // [T][D]
    unsigned long long *ldbar = reinterpret_cast<unsigned long long *>(xpart + T * D);
    const unsigned tid = threadIdx.x;
    const unsigned base = p.shard_begin + blockIdx.x * p.per_cta;
    const unsigned cnt = base >= p.shard_end ? 0u : min(p.per_cta, p.shard_end - base);
    const unsigned shard_size = p.shard_end - p.shard_begin;
    const unsigned ngroups = (cnt + T - 1) / T;
    if (tid == 0) kbar_init(ldbar, 1);
    __syncthreads();
    unsigned ldphase = 0, gcount = 0;

    DrawRec dr;
    auto make_draw = [&](long long h, unsigned l) {
        unsigned j;
        double z, u;
        step_draws<false>(p, h, base + l, j, z, u);
        dr.j = j;
        dr.z = z;
        dr.q = filter_q<false>(p, z, u);
    };
    if (tid < cnt) make_draw(p.h0, tid);

    ThinClock<> clk{p.n0, p.phase0, p.sidx0};
    unsigned long long target = p.bar_base;
    for (long long h = p.h0; h < p.h1; ++h) {
        const unsigned batch = (unsigned)(h & 1);
        const bool store = clk.store();
        const size_t a0 = batch ? (size_t)p.nhalf : 0;
        for (unsigned g = 0; g < ngroups; ++g, ++gcount) {
            const unsigned rows = min(T, cnt - g * T);
            const unsigned l = g * T + tid;
            const bool live = tid < rows;
            double *own = xown + (size_t)(gcount & 1) * T * D;
            if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");  // store of 2 groups ago read its buffer
            __syncthreads();                                                             // and everyone is done with xpart
            if (tid == 0) {
                kbar_expect_tx(ldbar, rows * ROWB * 2);
                bulk_row_g2s(own, p.x + (a0 + base + (size_t)g * T) * D, rows * ROWB, ldbar);
            }
            if (g > 0 && live) make_draw(h, l);
            if (live) {
                const unsigned pos = dr.j >= p.nhalf ? dr.j - p.nhalf : dr.j;
                const double *src = (PEER ? p.peer_x[pos / shard_size] : p.x) + (size_t)dr.j * D;
                bulk_row_g2s(xpart + (size_t)tid * D, src, ROWB, ldbar);
            }
            const size_t k = a0 + base + l;
            const double lpk = live ? p.lp[k] : 0.0;
            kbar_wait(ldbar, ldphase);
            ldphase ^= 1;
            if (live) {
                double xk[D], xj[D], y[D];
#pragma unroll
                for (int c = 0; c < D; c += 2) {
                    const double2 a2 = *reinterpret_cast<const double2 *>(own + (size_t)tid * D + c);
                    const double2 b2 = *reinterpret_cast<const double2 *>(xpart + (size_t)tid * D + c);
                    xk[c] = a2.x;
                    xk[c + 1] = a2.y;
                    xj[c] = b2.x;
                    xj[c + 1] = b2.y;
                }
                const double z = dr.z;
#pragma unroll
                for (int c = 0; c < D; ++c) y[c] = stretch_coord(xj[c], xk[c], z);  // :255
                const double p1 = dn.logpdf(y);                                      // :257
                const double tt = (p1 - lpk) + (double)dr.q * 0.6931471805599453;   // :260
                bool acc;
                if (tt > (double)p.margin) acc = true;
                else if (tt < -(double)p.margin) acc = false;
                else acc = accept_slow<false, false>(p, h, base + l, z, p1, lpk);
                if (acc) {  // :261-265
#if KMC_BULK_STORE_ALL
#pragma unroll
                    for (int c = 0; c < D; c += 2)
                        *reinterpret_cast<double2 *>(own + (size_t)tid * D + c) = make_double2(y[c], y[c + 1]);
#else
                    store_row<D>(p.x + k * D, y);
#endif
                    p.lp[k] = p1;
                    p.nacc[k] += 1u;
                }
                if (store) chain_store<D>(p, chain_row(p, clk.sidx, batch, base + l), acc, y, xk, p1, lpk);
            }
#if KMC_BULK_STORE_ALL
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // smem writes -> bulk store
            __syncthreads();
            if (tid == 0) bulk_s2g(p.x + (a0 + base + (size_t)g * T) * D, own, rows * ROWB);
#endif
        }
        if (batch == 1) {
            if (clk.burnin_end()) {  // :285-288
                for (unsigned l = tid; l < cnt; l += T) {
                    p.nacc[base + l] = 0u;
                    p.nacc[(size_t)p.nhalf + base + l] = 0u;
                }
            }
            clk.advance(store, p.nthin);
        }
#if KMC_BULK_STORE_ALL
        if (tid == 0) {  // all of this CTA's row stores are complete and ordered before the barrier
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            asm volatile("fence.proxy.async;" ::: "memory");
        }
#else
        asm volatile("fence.proxy.async;" ::: "memory");  // this thread's row stores (generic proxy) before the other CTAs' bulk gathers
#endif
        if (h + 1 < p.h1) {
            target += gridDim.x;
            __syncthreads();
            if (gridDim.x > 1 && tid == 0) barrier_arrive(p.barrier);
            if (tid < cnt) make_draw(h + 1, tid);  // first group of the next half-step, in the barrier's shadow
            if (gridDim.x > 1) {
                if (tid == 0) barrier_wait(p.barrier, target);
                __syncthreads();
            }
#if !KMC_BULK_STORE_ALL
            asm volatile("fence.proxy.async;" ::: "memory");  // acquired row stores -> this thread's bulk gathers
#endif
            if constexpr (PEER) {
                if (blockIdx.x == 0) cross_gpu_barrier(p, p.epoch_base + (unsigned long long)(h - p.h0) + 1);
                target += gridDim.x;
                __syncthreads();
                if (gridDim.x > 1) {
                    if (tid == 0) {
                        barrier_arrive(p.barrier);
                        barrier_wait(p.barrier, target);
                    }
                    __syncthreads();
                }
            }
        }
    }
}

// ------------------------------------------------------------------ shared-memory-resident kernel
// x / logp / accept counters of the CTA's walkers live in shared memory for the whole launch;
// global x is only written on accept (so partners can gather it) and logp / counters are
// written back once at the end.  Every thread owns at most kRounds walker positions of each
// half: slot(half b, round q) = b*per_cta + q*blockDim + tid.  Layout (L = 2*per_cta slots),
// component-major so that a warp's accesses are conflict-free:
//   double xs[D][L]; double lps[L]; unsigned naccs[L];
// Per half-step: the draws (Philox) of the first kSmemSplit rounds are made in the grid barrier's shadow, the others
// right after the first partner gathers are issued (under their L2 latency); partner rows are prefetched two rounds
// ahead.  Thread 0 arrives (release), the last warp polls (acquire loads).
// Geometry and split were swept on a B200 for the 2^20-walker config (us per half-step, profiles/r2_k1_variants_*.log):
// round 1 form (all draws in the shadow) 384x5x2 7.30; split 2: 384x5x2 6.85, 320x6x2 6.73, 256x7x2 6.65 (1771 positions
// per CTA = 6.92 x 256: every round full), 224x8x2 7.07, 192x10x2 7.67, 128x14x2 9.75, 448x4x2 7.70 (72-register cap),
// 256x5x3 9.64, 512x7x1 6.75; 256x7x2 with split 1 / 3 / 4 / 5 / 7: 6.89 / 6.48 / 6.52 / 6.69 / 7.57; + last warp
// polls: split 3 / 4 / 5 = 6.40 / 6.37 / 6.53; + acquire polls instead of relaxed polls and a fence: split 4 / 5 / 6 =
// 6.02 / 6.14 / 6.32.  Measured without gain: 3 partner rows in flight, two polls in flight, next round's own row
// preloaded, two rounds' proposals and log-densities interleaved per thread, per-warp arrivals (12x the atomics: 7.66),
// draws made inside the round loop (7.45), bit-assembled uniforms instead of I2F.F64.U64.
#ifndef KMC_SMEM_ROUNDS
#define KMC_SMEM_ROUNDS 7
#endif
#ifndef KMC_SMEM_THREADS
#define KMC_SMEM_THREADS 256
#endif
#ifndef KMC_SMEM_CTAS
#define KMC_SMEM_CTAS 2
#endif
#ifndef KMC_SMEM_SPLIT
#define KMC_SMEM_SPLIT 4
#endif
constexpr int kRounds = KMC_SMEM_ROUNDS;
constexpr int kSmemSplit = KMC_SMEM_SPLIT;  // draws of rounds [0, split) in the barrier's shadow, the rest after it (>= 2)
#ifndef KMC_SMEM_AHEAD
#define KMC_SMEM_AHEAD 2
#endif
constexpr int kAhead = KMC_SMEM_AHEAD;  // partner rows in flight per thread
static_assert(kSmemSplit >= kAhead && kSmemSplit <= kRounds, "the first partner gathers need their draws");
constexpr int kSmemThreads = KMC_SMEM_THREADS;
constexpr int kSmemCtas = KMC_SMEM_CTAS;  // CTAs per SM the kernel is compiled and launched for

// Shared memory through explicit 32-bit addresses: every access is (per-thread base) +
// (warp-uniform offset), so a thread keeps ONE address register for all of its slots.
__device__ __forceinline__ double lds_f64(unsigned a) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_f64(unsigned a, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory");
}
__device__ __forceinline__ unsigned lds_u32(unsigned a) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_u32(unsigned a, unsigned v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

template <template <int> class Dn, int D, bool REPLAY>
static __global__ void __launch_bounds__(kSmemThreads, kSmemCtas) emcee_smem_kernel(const RunParams p, const Dn<D> dn) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const unsigned nthr = blockDim.x;
    const unsigned L = 2 * p.per_cta;
    // ---- the per-thread registers that live across the whole launch -------------------
    const unsigned wid = p.shard_begin + blockIdx.x * p.per_cta + threadIdx.x;  // owned position of round 0 (in each half)
    const unsigned sbase = (unsigned)__cvta_generic_to_shared(smem_raw) + 8u * threadIdx.x;  // xs/lps slot of round 0
    const unsigned nbase = (unsigned)__cvta_generic_to_shared(smem_raw) + 8u * (D + 1) * L + 4u * threadIdx.x;
    double *const grow = p.x + (size_t)wid * D;  // own global row of (half 0, round 0)
    unsigned nv;                                 // rounds this thread owns (<= kRounds)
    {
        const unsigned base = p.shard_begin + blockIdx.x * p.per_cta;
        const unsigned cnt = base >= p.shard_end ? 0u : min(p.per_cta, p.shard_end - base);
        nv = cnt > threadIdx.x ? (cnt - threadIdx.x + nthr - 1) / nthr : 0u;
    }
    // slot(half b, round q) = b*per_cta + q*nthr (+ tid, folded into the bases); byte offsets
    // of x component c: 8*(c*L + slot), logp: 8*(D*L + slot), counter: 4*slot  -- all warp-uniform

    for (unsigned b = 0; b < 2; ++b)  // stage the owned walkers of both halves
        for (unsigned q = 0; q < nv; ++q) {
            const size_t ro = (size_t)b * p.nhalf + (size_t)q * nthr;
            const unsigned sl = b * p.per_cta + q * nthr;
            double v[D];
            load_row<D>(grow + ro * D, v);
#pragma unroll
            for (int c = 0; c < D; ++c) sts_f64(sbase + 8u * (c * L + sl), v[c]);
            sts_f64(sbase + 8u * (D * L + sl), p.lp[wid + ro]);
            sts_u32(nbase + 4u * sl, p.nacc[wid + ro]);
        }
    // a thread only ever touches the slots it staged itself: no sync needed

    DrawRec dr[kRounds];
    auto make_draws = [&](long long h, auto lo, auto hi) {  // rounds [lo, hi) of half-step h
#pragma unroll
        for (int q = decltype(lo)::value; q < decltype(hi)::value; ++q)
            if (q < nv) {
                unsigned j;
                double z, u;
                step_draws<REPLAY>(p, h, wid + q * nthr, j, z, u);  // :250, :252, (:260 uniform)
                dr[q].j = j;
                dr[q].z = z;
                dr[q].q = filter_q<REPLAY>(p, z, u);
            }
    };
    using SplitLo = std::integral_constant<int, 0>;
    using SplitMid = std::integral_constant<int, kSmemSplit>;
    using SplitHi = std::integral_constant<int, kRounds>;
    make_draws(p.h0, SplitLo{}, SplitMid{});

    // launch-local 32-bit bookkeeping of the reference's n (:245), rem(n, nthin) and the sample index
    const unsigned nh = (unsigned)(p.h1 - p.h0);
    ThinClock<unsigned> clk{p.n0, (unsigned)p.phase0, p.sidx0};
    unsigned long long target = p.bar_base;
    for (unsigned hh = 0; hh < nh; ++hh) {
        const long long h = p.h0 + hh;
        const unsigned batch = (unsigned)(h & 1);
        const bool store = clk.store();
        const unsigned hslot = batch ? p.per_cta : 0u;            // first slot of the active half
        const size_t hrow = batch ? (size_t)p.nhalf : (size_t)0;  // first global row of the active half (:247)

        double xj[kAhead][D];
#pragma unroll
        for (int q = 0; q < kAhead; ++q)
            if (q < nv) load_row_cg<D>(p.x + (size_t)dr[q].j * D, xj[q]);
        make_draws(h, SplitMid{}, SplitHi{});  // the later rounds' draws, under the first gathers' L2 latency
#pragma unroll
        for (int q = 0; q < kRounds; ++q) {
            if (q >= nv) break;
            const unsigned sl = hslot + q * nthr;      // warp-uniform
            const size_t ro = hrow + (size_t)q * nthr;  // warp-uniform
            double xk[D], y[D];
#pragma unroll
            for (int c = 0; c < D; ++c) xk[c] = lds_f64(sbase + 8u * (c * L + sl));
            const double lpk = lds_f64(sbase + 8u * (D * L + sl));
            const double z = dr[q].z;
#pragma unroll
            for (int c = 0; c < D; ++c) y[c] = stretch_coord(xj[q % kAhead][c], xk[c], z);  // :255
            if (q + kAhead < kRounds && q + kAhead < nv)  // partner row kAhead rounds ahead, before this round's stores
                load_row_cg<D>(p.x + (size_t)dr[(q + kAhead) % kRounds].j * D, xj[q % kAhead]);
            const double p1 = dn.logpdf(y);                                        // :257
            const double tt = (p1 - lpk) + (double)dr[q].q * 0.6931471805599453;  // :260
            bool acc;
            if (tt > (double)p.margin) acc = true;
            else if (tt < -(double)p.margin) acc = false;
            else acc = accept_slow<REPLAY, (D == 1 && !REPLAY)>(p, h, wid + q * nthr, z, p1, lpk);
            if (acc) {  // :261-265
                store_row<D>(grow + ro * D, y);
#pragma unroll
                for (int c = 0; c < D; ++c) sts_f64(sbase + 8u * (c * L + sl), y[c]);
                sts_f64(sbase + 8u * (D * L + sl), p1);
                sts_u32(nbase + 4u * sl, lds_u32(nbase + 4u * sl) + 1u);
            }
            if (store) chain_store<D>(p, chain_row(p, clk.sidx, batch, wid + q * nthr), acc, y, xk, p1, lpk);
        }
        if (batch == 1) {
            if (clk.burnin_end())  // :285-288 burn-in counters are discarded
                for (unsigned q = 0; q < nv; ++q) {
                    sts_u32(nbase + 4u * (q * nthr), 0u);
                    sts_u32(nbase + 4u * (p.per_cta + q * nthr), 0u);
                }
            clk.advance(store, (unsigned)p.nthin);
        }
        if (hh + 1 < nh)  // the draws in the barrier's shadow are independent of the other CTAs
            grid_join<true>(p, target, [&] { make_draws(h + 1, SplitLo{}, SplitMid{}); });
    }

    for (unsigned b = 0; b < 2; ++b)  // write back what only lived in shared memory
        for (unsigned q = 0; q < nv; ++q) {
            const size_t ro = (size_t)b * p.nhalf + (size_t)q * nthr;
            const unsigned sl = b * p.per_cta + q * nthr;
            p.lp[wid + ro] = lds_f64(sbase + 8u * (D * L + sl));
            p.nacc[wid + ro] = lds_u32(nbase + 4u * sl);
        }
}

// K4: batched log-density (initial p0s, src/samplers.jl:209; make_theta0s, :334-338).
template <template <int> class Dn, int D>
static __global__ void __launch_bounds__(256) density_eval_kernel(const double *__restrict__ x, double *__restrict__ out,
                                                           long long nw, const Dn<D> dn) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nw) return;
    double v[D];
    load_row<D>(x + w * D, v);
    out[w] = dn.logpdf(v);
}

// Chain store is sample-major on the device ([ns][nw][D]); the ABI wants walker-major
// ([nw][ns][D]).  Transposes walkers [w0, w0+wc), samples [s0, s0 + 32*gridDim.y) into a staging buffer.
// INDEXED: walker w is stored row idx[w] (squash's kept walkers); else row w.
constexpr long long kTransposeMaxSamples = 65535LL * 32;  // gridDim.y limit: longer chains take several launches
template <bool INDEXED>
static __global__ void chain_transpose_kernel(const double *__restrict__ in, double *__restrict__ out, long long ns,
                                       long long nw, long long w0, long long wc, int d, long long s0,
                                       const unsigned *__restrict__ idx) {
    __shared__ double tile[32][33];
    // element (s, w) is a d-vector; handle one component per blockIdx.z
    const int c = blockIdx.z;
    const long long wb = (long long)blockIdx.x * 32, sb = s0 + (long long)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const long long s = sb + r, w = wb + threadIdx.x;
        if (s < ns && w < wc) tile[r][threadIdx.x] = in[(s * nw + (INDEXED ? (long long)idx[w0 + w] : w0 + w)) * d + c];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const long long w = wb + r, s = sb + threadIdx.x;
        if (s < ns && w < wc) out[(w * ns + s) * d + c] = tile[threadIdx.x][r];
    }
}

// Posterior moments of the stored chain on the device (the squash_walkers + mean/var reduction
// of src/samplers.jl:372-428 + test/runtests.jl:36-43 without copying the chain to the host):
// per component, sum and sum of squares of (x - shift), shift = the first stored sample.
static __global__ void __launch_bounds__(256) chain_moments_kernel(const double *__restrict__ chain, long long nrows, int d,
                                                            double *__restrict__ sums /* [2][d] */) {
    extern __shared__ double sh[];  // [2][d]
    for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) sh[c] = 0.0;
    __syncthreads();
    const long long total = nrows * d;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(e % d);
        const double v = chain[e] - chain[c];
        atomicAdd(&sh[c], v);
        atomicAdd(&sh[d + c], v * v);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) atomicAdd(&sums[c], sh[c]);
}

// K5: accept-counter statistics of the progress display (src/samplers.jl:276-278).
static __global__ void nacc_sum_kernel(const unsigned *__restrict__ nacc, long long nw, unsigned long long *sum) {
    unsigned long long s = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += (long long)gridDim.x * blockDim.x)
        s += nacc[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(sum, s);
}

static __global__ void nacc_moment_kernel(const unsigned *__restrict__ nacc, long long nw, double mean, double thresh,
                                   double *ssq, unsigned long long *outl) {
    double s = 0.0;
    unsigned long long o = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += (long long)gridDim.x * blockDim.x) {
        const double dv = (double)nacc[i] - mean;
        s += dv * dv;
        o += (thresh >= 0.0 && fabs(dv) > thresh) ? 1 : 0;
    }
    for (int k = 16; k > 0; k >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, k);
        o += __shfl_xor_sync(0xffffffffu, o, k);
    }
    if ((threadIdx.x & 31) == 0) {
        if (ssq) atomicAdd(ssq, s);
        if (outl && o) atomicAdd(outl, o);
    }
}

}  // namespace kmc
